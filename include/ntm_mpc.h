/* ntm_mpc.h -- C ABI of the B200-native LPV-MPC hot path (libntm_mpc.so).
 *
 * Drop-in boundary for the MATLAB functions that IsaacSavona/MPC-NTM-Control resolves by name on the
 * path (citations relative to the upstream tree).  Every entry point is `extern "C"`, takes plain
 * pointers and sizes, returns an int status (0 = NTM_OK) and never throws; ntm_last_error() returns the
 * message of the last failure on the calling thread.  A handle owns one CUDA device, one stream and
 * its scratch buffers; it is not thread-safe (one handle per host thread / per GPU).
 *
 * An argument error returns NTM_ERR_INVALID before anything is allocated, copied or launched.
 *
 * There is NO CPU fallback: every compute entry point launches hand-written sm_100a kernels and
 * fails with NTM_ERR_CUDA when no CUDA device is usable.
 *
 * Two pointer flavours per operation:
 *   ntm_xxx      host pointers; inputs are copied H2D and results D2H inside the call (blocking).
 *   ntm_xxx_dev  device pointers; asynchronous on the handle's stream (ntm_set_stream / ntm_sync).
 *
 * Layouts (argument `layout`), for an array holding a block of E doubles per scenario, S scenarios:
 *   NTM_LAYOUT_MATLAB  element e of scenario s at [s*E + e]  -- what MATLAB holds for a (.., .., S) array,
 *                      each block column-major exactly as the reference function returns it.
 *   NTM_LAYOUT_SOA     element e of scenario s at [e*S + s]  -- scenario index fastest.
 * Inside a block the element order is always MATLAB column-major:
 *   x (2x1): [w, omega];  A (2x2): [a11,a21,a12,a22];  B (2x1): [b,0];
 *   Phi (2N x 2), Gamma (2N x N), Lambda (2N x 1), G (N x N), F (N x 1), U (N x 1),
 *   xk (2 x (k_sim+1)), uk (1 x k_sim), Uk (N x k_sim).
 *
 * Parameter block (`params`, NTM_NPARAM doubles per scenario, same layout rule; `params_count` is S, or 1
 * to broadcast one block to all scenarios).  Hoisted coefficients of A.m:2 / B.m:2 / NTM_MPC_Sim.m:37:
 *   [0] c_a11 = (4/3)*(kappa*rs/(0.82*taur))*Ts      a11 = c_a11*rho1 + 1            (A.m:2)
 *   [1] c_a21 = Ts/(zeta*a^3)                        a21 = c_a21*rho2                (A.m:2)
 *   [2] a22   = 1 - Ts/TE                                                            (A.m:2)
 *   [3] c_b   = kappa*Ts*etaCD/wdep                  b   = c_b*rho3                  (B.m:2)
 *   [4] C1, [5] C2                                   affine term                     (NTM_MPC_Sim.m:37)
 *   [6] wmarg2 = w_marg^2                            rho1                            (rho1.m:2)
 *   [7] w_dep                                        rho3                            (rho3.m:2)
 *   [8] umin, [9] umax                               EC-power box                    (NTM_MPC_Sim.m:47-50)
 *   [10] r1, [11] r2                                 reference state                 (NTM_MPC_Sim.m:60)
 *   [12] q11, [13] q12, [14] q22                     Q                               (NTM_MPC_Sim.m:59)
 *   [15] c_tauE [1/m]                               tau_E(w) = tau_E0*(1 - c_tauE*w), read only with NTM_PROFILE_TAUE_W
 *                                                    (NTM_MPC_Sim.m:14 "NOT EXACT FORMULA"); 0 otherwise
 */
#ifndef NTM_MPC_H
#define NTM_MPC_H

#ifdef __cplusplus
extern "C" {
#endif

#define NTM_VERSION 100 /* 0.1.0 */
#define NTM_NPARAM 16
#define NTM_MAX_HORIZON 128

/* status codes returned by every function */
enum {
    NTM_OK = 0,
    NTM_ERR_INVALID = 1, /* bad argument (NULL, size out of range, unknown layout) */
    NTM_ERR_CUDA = 2,    /* CUDA runtime/driver failure, or no device: there is no CPU fallback */
    NTM_ERR_ALLOC = 3
};

/* per-scenario status words written by the QP and closed-loop kernels (max over the run) */
enum {
    NTM_SCN_OK = 0,
    NTM_SCN_QP_ITER_CAP = 1,  /* pivoting iteration cap reached (solution still projected onto the box) */
    NTM_SCN_NONFINITE = 2,    /* non-finite state, Hessian or solution (IEEE propagation, no fast-math) */
    NTM_SCN_INFEASIBLE = 3    /* ntm_qp_ineq: no U satisfies the rows (quadprog exitflag -2, NTM_MPC_Sim.m:100-101) */
};

enum { NTM_LAYOUT_MATLAB = 0, NTM_LAYOUT_SOA = 1 };

/* profile switches (SURVEY 2.4); 0 = the literal, minimally repaired reading of the reference */
enum {
    NTM_PROFILE_RHO1_SQ = 1,      /* rho1 = 1/(w^2 + w_marg^2)  (rhos.m:18) instead of rho1.m:2 */
    NTM_PROFILE_GAMMA_I = 2,      /* Gamma(i,j) = A_i*Gamma(i-1,j) instead of A_{i-j} (Rho_to_PhiGammaLambda.m:32) */
    NTM_PROFILE_F_XK = 4,         /* F built from xk(:,k) instead of x0 (NTM_MPC_Sim.m:73,121) */
    NTM_PROFILE_PLANT_C = 8,      /* plant step adds +C (NTM_MPC_Sim.m:130 omits it) */
    NTM_PROFILE_INNER_FIXED = 16, /* always run i_sim inner iterations (no 1e-14 break, NTM_MPC_Sim.m:123-126) */
    NTM_PROFILE_DENSE_G = 32,     /* diagnostic: force the dense row-sweep G/F build even where the literal
                                     Gamma has the Toeplitz structure the fast path uses (same result) */
    NTM_PROFILE_PLANT_RK4 = 64,   /* fidelity option (SURVEY 8f-4), NOT the reference: NTM_MPC_Sim.m:130 is the forward-
                                     Euler map x+ = x + g(x,u), g = (A(rho(x))-I)x + B(rho(x))u (+C); this bit integrates
                                     dx/dt = g(x,u)/Ts over one sample with the classical 4-stage Runge-Kutta scheme,
                                     u held.  The controller's prediction model is unchanged. */
    NTM_PROFILE_TAUE_W = 128      /* fidelity hook (SURVEY 8f-4), NOT the reference: NTM_MPC_Sim.m:14 sets tau_E = tau_E0
                                     and marks it "currently NOT EXACT FORMULA".  With this bit the energy confinement
                                     time degrades with the island width, tau_E(w) = tau_E0*(1 - c_tauE*w) (params[15];
                                     the belt model of Chang & Callen gives c_tauE = 4 rs^3/a^4), i.e. the (2,2) entry of
                                     A.m:2 becomes a22(w) = 1 - (1 - a22)/(1 - c_tauE*w).  ntm_plant_step evaluates it at
                                     the state it is given (every RK4 stage at its own); the closed loop re-evaluates it
                                     from the MEASURED width xk(1,k) at the top of each time step and holds it over the
                                     prediction horizon of that step (the rho's vary along the horizon, tau_E does not:
                                     G, F on hand from the previous step keep the previous value).  The per-call entry
                                     points take tau_E through params[2] exactly like A.m takes TE. */
};
#define NTM_PROFILE_LITERAL 0
#define NTM_PROFILE_CONSISTENT (NTM_PROFILE_GAMMA_I | NTM_PROFILE_F_XK | NTM_PROFILE_PLANT_C)

typedef struct ntm_handle ntm_handle;

/* ---- lifetime ---------------------------------------------------------------------------- */
int ntm_create(ntm_handle **out, int device);          /* device = CUDA ordinal */
int ntm_destroy(ntm_handle *h);
/* A handle works on ONE stream at a time (its scratch buffers and work queue are shared by everything queued through
 * it): both calls below first synchronise the stream being left.  *_dev entry points are asynchronous except that the
 * first call for a longer horizon N (and host entries whose staging arena grows) synchronise and allocate scratch. */
int ntm_set_stream(ntm_handle *h, void *cuda_stream);  /* cudaStream_t of the caller; NULL = the legacy default stream */
int ntm_reset_stream(ntm_handle *h);                   /* back to the handle's own non-blocking stream */
int ntm_sync(ntm_handle *h);
const char *ntm_last_error(void);
int ntm_version(void);
/* sm_count, compute capability and the number of kernel launches issued through this handle so far */
int ntm_device_info(ntm_handle *h, int *sm_count, int *cc_major, int *cc_minor);
long long ntm_launch_count(ntm_handle *h);

/* ---- rho1.m:1-3, rho2.m:1-3, rho3.m:1-4 (variant rhos.m:17-19) ---------------------------- *
 * x[2*S] -> rho1[S], rho2[S], rho3[S].  Replaces the calls at NTM_MPC_Sim.m:63-65,114-116,130.   */
int ntm_rho(ntm_handle *h, int layout, int profile, int S, const double *x, const double *params,
            int params_count, double *rho1, double *rho2, double *rho3);
int ntm_rho_dev(ntm_handle *h, int layout, int profile, int S, const double *x, const double *params,
                int params_count, double *rho1, double *rho2, double *rho3);

/* ---- A.m:1-3, B.m:1-3 --------------------------------------------------------------------- *
 * rho1..3[S] -> A[4*S] (2x2 column-major), B[2*S] (the 2x1 column [b;0], defect D7).              */
int ntm_lpv_AB(ntm_handle *h, int layout, int S, const double *rho1, const double *rho2, const double *rho3,
               const double *params, int params_count, double *A, double *B);
int ntm_lpv_AB_dev(ntm_handle *h, int layout, int S, const double *rho1, const double *rho2, const double *rho3,
                   const double *params, int params_count, double *A, double *B);

/* ---- Rho_to_PhiGammaLambda.m:1-54 --------------------------------------------------------- *
 * Rho1..3[N*S] -> Phi[4N*S], Gamma[2N*N*S], Lambda[2N*S].  profile: NTM_PROFILE_GAMMA_I selects the
 * index of line :32.  1 <= N <= NTM_MAX_HORIZON.                                                  */
int ntm_condense(ntm_handle *h, int layout, int profile, int S, int N, const double *Rho1, const double *Rho2,
                 const double *Rho3, const double *params, int params_count, double *Phi, double *Gamma,
                 double *Lambda);
int ntm_condense_dev(ntm_handle *h, int layout, int profile, int S, int N, const double *Rho1, const double *Rho2,
                     const double *Rho3, const double *params, int params_count, double *Phi, double *Gamma,
                     double *Lambda);

/* ---- NTM_MPC_Sim.m:67-73,120-121 ---------------------------------------------------------- *
 * G = 2*Gamma'*Omega*Gamma (N x N), F = 2*Gamma'*Omega*(Phi*x + Lambda - R) (N), Omega = I_N (x) Q,
 * R = repmat(r(:),N,1); Q and r come from the parameter block.  Gamma may be any dense 2N x N matrix. */
int ntm_hessian_grad(ntm_handle *h, int layout, int S, int N, const double *Phi, const double *Gamma,
                     const double *Lambda, const double *x, const double *params, int params_count, double *G,
                     double *F);
int ntm_hessian_grad_dev(ntm_handle *h, int layout, int S, int N, const double *Phi, const double *Gamma,
                         const double *Lambda, const double *x, const double *params, int params_count,
                         double *G, double *F);

/* ---- quadprog(G,F,...) with only the input-box rows of getWLc.m:14-23 (NTM_MPC_Sim.m:97) --- *
 * min 1/2 U'GU + F'U  s.t. lb <= U <= ub, G symmetric positive definite.  lb/ub hold N doubles per
 * scenario (bounds_count = S) or one shared block (bounds_count = 1).  iters[S], status[S] may be NULL. */
int ntm_qp_box(ntm_handle *h, int layout, int S, int N, const double *G, const double *F, const double *lb,
               const double *ub, int bounds_count, double *U, int *iters, int *status);
int ntm_qp_box_dev(ntm_handle *h, int layout, int S, int N, const double *G, const double *F, const double *lb,
                   const double *ub, int bounds_count, double *U, int *iters, int *status);

/* ---- quadprog(G,F,L,c+W*x) as NTM_MPC_Sim.m:97 calls it, state rows of getWLc.m:11-12,25 kept --- *
 * min 1/2 U'GU + F'U  s.t. lb <= U <= ub (finite, as getWLc.m:14-23 always provides) and Lg*U <= bg, Lg M x N
 * per scenario (MATLAB layout: column-major M x N blocks, scenario slowest), bg[M*S].  The host side of a quadprog
 * shim splits the rows of L: one non-zero -> a bound, all zero -> feasibility of the right-hand side, the rest ->
 * Lg (csrc/mex/ntm_mex.c gateway 10, ntm_mpc.reference_api.quadprog).  status: NTM_SCN_OK, NTM_SCN_QP_ITER_CAP,
 * NTM_SCN_NONFINITE or NTM_SCN_INFEASIBLE (quadprog exitflag 1 / 0 / -- / -2).  M = 0 is ntm_qp_box.  Needs both
 * N x N factors in shared memory: N <= ~100 on a B200, NTM_ERR_INVALID beyond. */
int ntm_qp_ineq(ntm_handle *h, int layout, int S, int N, int M, const double *G, const double *F, const double *lb,
                const double *ub, int bounds_count, const double *Lg, const double *bg, double *U, int *iters,
                int *status);
int ntm_qp_ineq_dev(ntm_handle *h, int layout, int S, int N, int M, const double *G, const double *F,
                    const double *lb, const double *ub, int bounds_count, const double *Lg, const double *bg,
                    double *U, int *iters, int *status);

/* ---- NTM_MPC_Sim.m:130 --------------------------------------------------------------------- *
 * x_next = A(rho(x))*x + B(rho(x))*u (+ C with NTM_PROFILE_PLANT_C); NTM_PROFILE_PLANT_RK4 replaces the Euler map by
 * one RK4 step of the same vector field.  x[2*S], u[S] -> x_next[2*S].   */
int ntm_plant_step(ntm_handle *h, int layout, int profile, int S, const double *x, const double *u,
                   const double *params, int params_count, double *x_next);
int ntm_plant_step_dev(ntm_handle *h, int layout, int profile, int S, const double *x, const double *u,
                       const double *params, int params_count, double *x_next);

/* ---- NTM_MPC_Sim.m:63-73 + 80-131: the whole closed loop, fused, batched over S scenarios --- *
 * x0[2*S], params -> xk[2*(k_sim+1)*S], uk[k_sim*S], Uk[N*k_sim*S] (NULL to skip), cost[S] (sum over the
 * closed-loop states k=1..k_sim of (x-r)'Q(x-r)), inner_iters[k_sim*S] (re-linearisations per step),
 * qp_iters[k_sim*S] (QP pivoting iterations per step), status[S].  Any output except xk/uk may be NULL. */
int ntm_mpc_closed_loop(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                        const double *x0, const double *params, int params_count, double *xk, double *uk,
                        double *Uk, double *cost, int *inner_iters, int *qp_iters, int *status);
int ntm_mpc_closed_loop_dev(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim,
                            double eps, const double *x0, const double *params, int params_count, double *xk,
                            double *uk, double *Uk, double *cost, int *inner_iters, int *qp_iters, int *status);

/* ---- the same loop with the state rows of getWLc.m:9-12,25 kept in every QP (SURVEY 8f-1) ------------------ *
 * NTM_MPC_Sim.m:97 passes L*U <= c + W*xk(:,k) to quadprog, L/W/c from getWLc (:74).  state_rows selects what the rows
 * are built from:
 *   NTM_STATE_ROWS_OFF      no state rows: identical to ntm_mpc_closed_loop (the EC-power box only).
 *   NTM_STATE_ROWS_REFRESH  rebuilt from every re-condensation (:119), i.e. the rows always describe the prediction
 *                           model the cost uses -- what a maintained script would do.
 *   NTM_STATE_ROWS_FROZEN   the literal reading: :74 sits outside both loops, so L, W, c keep the offline build
 *                           (rho(x0) on every stage, :63-66) for the whole run while G and F are refreshed.
 * xbounds = {xmin(1), xmax(1), xmin(2), xmax(2)} on the HOST (NTM_MPC_Sim.m:44-45, shared by all scenarios).  No L
 * is ever stored: with the literal Gamma the rows are generated on the fly from its Toeplitz structure (any horizon
 * whose two N x N factors + 4N rows of bookkeeping fit shared memory, N <= ~100, NTM_ERR_INVALID beyond); with
 * NTM_PROFILE_GAMMA_I / DENSE_G they are read from the dense Gamma tile the tensor-core Hessian build keeps in shared
 * memory (getWLc.m:57 on the Gamma of Rho_to_PhiGammaLambda.m:32 index i; one-warp groups: N <= 32, NTM_ERR_INVALID
 * beyond).  The x_0 block (getWLc.m:30) makes a QP infeasible as soon as xk(:,k) itself leaves the state box.
 * An infeasible QP (quadprog exitflag -2, :100-101: no U comes back and the script cannot continue) ends the scenario:
 * status = NTM_SCN_INFEASIBLE, uk, xk and Uk from that step on and cost are NaN, inner_iters[k] = the iteration that
 * failed, 0 afterwards. */
enum { NTM_STATE_ROWS_OFF = 0, NTM_STATE_ROWS_REFRESH = 1, NTM_STATE_ROWS_FROZEN = 2 };
int ntm_mpc_closed_loop_sc(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                           const double *x0, const double *params, int params_count, int state_rows,
                           const double *xbounds, double *xk, double *uk, double *Uk, double *cost, int *inner_iters,
                           int *qp_iters, int *status);
int ntm_mpc_closed_loop_sc_dev(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                               const double *x0, const double *params, int params_count, int state_rows,
                               const double *xbounds, double *xk, double *uk, double *Uk, double *cost,
                               int *inner_iters, int *qp_iters, int *status);

/* ---- one receding-horizon step of the same controller, no plant (NTM_MPC_Sim.m:94-128): the caller closes the loop ---- *
 * For S scenarios at their measured states x[2*S] (xk(:,k)), runs the inner re-linearisation loop of one time step and
 * returns u[S] = uk(k) = U(1) (:107), U[N*S] = Uk(:,k), the last QP solution of the step (:106), inner_iters[S] and
 * qp_iters[S] as in ntm_mpc_closed_loop, and status[S]: the worst QP status of this step, NTM_SCN_NONFINITE if x or u is
 * not finite.  U, inner_iters, qp_iters and status may be NULL.  x, u and U follow `layout`.
 * state holds NTM_CTRL_DOUBLES(N) doubles per scenario, one contiguous record per scenario in both layouts, read and
 * written in place (host entry: copied in and back; _dev entry: resident on the device).  An ALL-ZERO record is a fresh
 * controller: its first step runs the offline build (:63-73) from rho(x) and x becomes the script's x0.  There is no
 * init call -- memset is the reset, and zeroing single records restarts single scenarios.  A record carries everything
 * that crosses a time step of the fused loop:
 *   [0, N)   a11   [N, 2N) a21   [2N, 3N) b      stage entries of the last re-scheduling (:114-117)
 *   [3N, 4N) Uold (:86,127, D13)                 [4N, 5N) and [5N, 6N): the last two QP solutions (warm starts)
 *   [6N, 7N) their partition states, (s1 + 1) + 4 (s2 + 1), s in {-1 lower, 0 free, +1 upper}
 *            (ntm_mpc_step_sc, literal Gamma: + 16 hw1 + 1024 hw2, see there)
 *   [7N, 7N+2) the last state this controller saw: the state the G, F on hand were built from under NTM_PROFILE_F_XK
 *   [7N+2, 7N+4) x0 (G, F of the literal profile)   [7N+4] cost (two-phase fused loop only)
 *   [7N+5] status + 4 first_qp + 8 n (n = warm-start history length, 3 = sticky "a warm QP ran long")
 *          (ntm_mpc_step_sc, literal Gamma: + 32 hwn, see there)
 *   [7N+6] steps this record has run (0 = fresh)
 * Preconditions (not checked by the kernel): every call for a record passes the same N, profile and params.
 * profile: every bit of the fused loop's box-QP instantiations (RHO1_SQ, GAMMA_I, DENSE_G, F_XK, INNER_FIXED); the
 * plant-only bits PLANT_C and PLANT_RK4 are accepted and ignored, so that one profile word drives both this entry and
 * ntm_plant_step; NTM_PROFILE_TAUE_W is rejected (NTM_ERR_INVALID).  1 <= N <= NTM_MAX_HORIZON, i_sim >= 1.  One step is
 * one kernel launch.  Stepped with ntm_plant_step under the same profile, k_sim steps reproduce ntm_mpc_closed_loop
 * bit for bit. */
#define NTM_CTRL_DOUBLES(N) (7 * (N) + 7)
int ntm_mpc_step(ntm_handle *h, int layout, int profile, int S, int N, int i_sim, double eps, const double *x,
                 const double *params, int params_count, double *state, double *u, double *U, int *inner_iters,
                 int *qp_iters, int *status);
int ntm_mpc_step_dev(ntm_handle *h, int layout, int profile, int S, int N, int i_sim, double eps, const double *x,
                     const double *params, int params_count, double *state, double *u, double *U, int *inner_iters,
                     int *qp_iters, int *status);

/* ---- the same step with getWLc's state rows kept in every QP: the controller NTM_MPC_Sim.m:97 solves ------------- *
 * ntm_mpc_step with state_rows and xbounds as in ntm_mpc_closed_loop_sc (xbounds on the HOST for both entries).
 * NTM_STATE_ROWS_OFF is ntm_mpc_step: the same launch and the same bits.  Stepped with ntm_plant_step under the same
 * profile, k_sim steps reproduce ntm_mpc_closed_loop_sc bit for bit, up to the step at which a scenario turns infeasible.
 * Infeasible step (quadprog exitflag -2, :100-101): u and U are NaN, status = NTM_SCN_INFEASIBLE, inner_iters and
 * qp_iters count that step as the fused loop does, and the record is NOT written: it still holds the controller as it
 * was before the call.  The caller decides: zero the record to restart, or call again with a new measurement.
 * Preconditions (not checked by the kernel): every call for a record passes the same N, profile, params, state_rows
 * and xbounds.  Record words beyond ntm_mpc_step's (literal Gamma; zero on every other path, so NTM_CTRL_DOUBLES(N)
 * is unchanged): the active sets of the last two state-row QPs, offered to the next QP as a warm start, per stage j
 * hw = (v + 1) + 4 m with v the variable's bound state and bit q of m = row 4j + q active; [6N + j] carries
 * 16 hw1 + 1024 hw2 and [7N+5] carries 32 hwn (hwn = how many of hw1, hw2 are valid, 0..2).  Frozen rows (:74) are
 * not stored: each resumed step rebuilds them from rho(x0) with x0 from [7N+2, 7N+4), one extra G, F build.
 * NTM_ERR_INVALID: NTM_PROFILE_TAUE_W, state_rows outside 0..2, NULL or inverted xbounds, GAMMA_I / DENSE_G with
 * N > 32, a horizon whose factors do not fit shared memory. */
int ntm_mpc_step_sc(ntm_handle *h, int layout, int profile, int S, int N, int i_sim, double eps, const double *x,
                    const double *params, int params_count, int state_rows, const double *xbounds, double *state,
                    double *u, double *U, int *inner_iters, int *qp_iters, int *status);
int ntm_mpc_step_sc_dev(ntm_handle *h, int layout, int profile, int S, int N, int i_sim, double eps, const double *x,
                        const double *params, int params_count, int state_rows, const double *xbounds, double *state,
                        double *u, double *U, int *inner_iters, int *qp_iters, int *status);

/* ---- the fused loop against a perturbed plant: the nominal controller, a plant it does not know exactly ---------- *
 * For k = 0 .. k_sim-1, with y_k the state the controller sees:
 *   y_k = x_k + v_k                          (measurement noise; v NULL: y_k = x_k)
 *   u_k, U_k = one ntm_mpc_step of the controller (profile, params, its own record) at y_k
 *   x_{k+1} = ntm_plant_step(x_k, u_k; plant_params, plant_profile) + d_k   (process disturbance; w NULL: none)
 * bit for bit, in ONE launch on the handle's stream.  xk(:,0) = x0 is the true initial state; the controller's offline
 * build (:63-73) runs from y_0.  xk holds the TRUE states, cost sums (x-r)'Q(x-r) over the true states k = 1..k_sim with
 * r and Q from the controller's block, status is the worst over the run (NTM_SCN_NONFINITE for a non-finite y, u or x).
 * Outputs as in ntm_mpc_closed_loop.  w (the disturbances d_k) and v: 2*k_sim doubles per scenario in `layout`, element
 * 2k + i, or NULL.  plant_params: NTM_NPARAM doubles per block in `layout`, plant_params_count 1 or S; NULL = params.
 * profile: what ntm_mpc_step takes (PLANT_C and PLANT_RK4 are ignored, TAUE_W is rejected).  plant_profile: exactly the
 * bits ntm_plant_step honours, RHO1_SQ | PLANT_C | PLANT_RK4 | TAUE_W (c_tauE from plant_params[15]).  With
 * plant_params = params, plant_profile = the plant bits of profile and w = v = NULL, every output is bit-identical to
 * ntm_mpc_closed_loop.  The controller solves the box QP; ntm_mpc_closed_loop_perturbed_sc below keeps getWLc's state
 * rows.  A controller-side tau_E(w) is not offered.
 * NTM_ERR_INVALID: bad sizes, NULL x0 / xk / uk / params, plant_params_count not 1 or S, a controller profile with
 * TAUE_W, a plant_profile bit outside the four above. */
int ntm_mpc_closed_loop_perturbed(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                                  const double *x0, const double *params, int params_count, const double *plant_params,
                                  int plant_params_count, int plant_profile, const double *w, const double *v,
                                  double *xk, double *uk, double *Uk, double *cost, int *inner_iters, int *qp_iters,
                                  int *status);
int ntm_mpc_closed_loop_perturbed_dev(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim,
                                      double eps, const double *x0, const double *params, int params_count,
                                      const double *plant_params, int plant_params_count, int plant_profile,
                                      const double *w, const double *v, double *xk, double *uk, double *Uk,
                                      double *cost, int *inner_iters, int *qp_iters, int *status);

/* ---- the same loop with getWLc's state rows kept in every QP: does the TRUE state stay inside the state box? ----- *
 * ntm_mpc_closed_loop_perturbed with state_rows and xbounds as in ntm_mpc_closed_loop_sc (xbounds on the HOST for both
 * entries).  For k = 0 .. k_sim-1, in ONE launch:
 *   y_k = x_k + v_k
 *   u_k, U_k = one ntm_mpc_step_sc (profile, params, state_rows, xbounds, its own record) at y_k
 *   x_{k+1} = ntm_plant_step(x_k, u_k; plant_params, plant_profile) + d_k
 * bit for bit, up to and including the step at which a scenario turns infeasible.  The offline build (:63-73) and the
 * frozen rows (:74) come from y_0; the x_0 block of getWLc.m:30 tests y_k, so measurement noise alone can make a QP
 * infeasible.  At the infeasible step u_k and U_k are NaN and inner_iters / qp_iters count the step as ntm_mpc_step_sc
 * does; from then on the scenario ends as in ntm_mpc_closed_loop_sc: uk, Uk and xk(:, k+1 ..) are NaN, the iteration
 * counts 0, cost NaN, status NTM_SCN_INFEASIBLE.  xk and cost are the true states, as in ntm_mpc_closed_loop_perturbed.
 * NTM_STATE_ROWS_OFF is ntm_mpc_closed_loop_perturbed (the same launch and the same bits).  With nothing perturbed
 * (plant_params NULL, plant_profile = the plant bits of profile, w = v = NULL) every output is bit-identical to
 * ntm_mpc_closed_loop_sc.  The plant's inputs travel to the kernel with its launch parameters: the _dev entry queues
 * the launch and no copy.
 * NTM_ERR_INVALID: whatever ntm_mpc_closed_loop_perturbed or ntm_mpc_step_sc rejects. */
int ntm_mpc_closed_loop_perturbed_sc(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim,
                                     double eps, const double *x0, const double *params, int params_count,
                                     int state_rows, const double *xbounds, const double *plant_params,
                                     int plant_params_count, int plant_profile, const double *w, const double *v,
                                     double *xk, double *uk, double *Uk, double *cost, int *inner_iters, int *qp_iters,
                                     int *status);
int ntm_mpc_closed_loop_perturbed_sc_dev(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim,
                                         double eps, const double *x0, const double *params, int params_count,
                                         int state_rows, const double *xbounds, const double *plant_params,
                                         int plant_params_count, int plant_profile, const double *w, const double *v,
                                         double *xk, double *uk, double *Uk, double *cost, int *inner_iters,
                                         int *qp_iters, int *status);

/* ---- state observer: one step of an LPV Kalman filter on the controller's own model, per scenario ---------------- *
 * The quasi-LPV Kalman filter: rho is frozen at the estimate, as the condensation (:63-66) freezes it; no Jacobian of
 * rho1..rho3 (not an EKF).  For S scenarios at the measurements y[2*S] (layout) and the inputs u[S] applied since their
 * last step, it updates each scenario's record in place and writes the estimate to xhat[2*S] (layout; may be NULL).
 * state holds NTM_KF_DOUBLES doubles per scenario, one contiguous record per scenario in both layouts:
 *   [0, 2) xhat   [2, 5) P as p11, p21, p22   [5] steps run (0 = fresh)
 * An ALL-ZERO record is a fresh filter (memset is the reset, as for NTM_CTRL_DOUBLES).  One step:
 *   fresh record:  xhat = y, P = Rv, steps = 1 (u is not read)
 *   otherwise:     xhat- = ntm_plant_step(xhat, u) under profile & (RHO1_SQ | PLANT_C | PLANT_RK4), params
 *                  F = A(rho(xhat)) of A.m:2 (the Euler-map matrix, also under PLANT_RK4: the quasi-LPV approximation)
 *                  P- = F P F' + Qw,  K = P- (P- + Rv)^-1 (closed-form 2x2 inverse),  xhat = xhat- + K (y - xhat-)
 *                  P = (I - K) P- (I - K)' + K Rv K' (Joseph form: P stays symmetric positive semi-definite although
 *                  w ~ 0.1 m and omega ~ 6e3 rad/s differ in scale by ~1e5),  steps += 1
 * Non-finite inputs get no special case: they propagate into the record, and zeroing it restarts the filter.
 * kf_cov = {qw11, qw21, qw22, rv11, rv21, rv22} on the HOST in both variants (shared by all scenarios): Qw the process
 * and Rv the measurement covariance.  profile: the controller's profile word (the other bits are ignored).  One launch.
 * host entry: records copied in and back; _dev entry: records resident.  u must be non-NULL for S > 0.
 * NTM_ERR_INVALID: NULL or non-finite kf_cov, Qw not positive semi-definite (q11 >= 0, q22 >= 0, q11 q22 >= q21^2), Rv
 * not positive definite (r11 > 0, r11 r22 > r21^2; then P- + Rv is invertible for every reachable P-), NTM_PROFILE_TAUE_W
 * in profile, bad sizes, NULL arrays, params_count not 1 or S. */
#define NTM_KF_DOUBLES 6
int ntm_kf_step(ntm_handle *h, int layout, int profile, int S, const double *y, const double *u, const double *params,
                int params_count, const double *kf_cov, double *state, double *xhat);
int ntm_kf_step_dev(ntm_handle *h, int layout, int profile, int S, const double *y, const double *u,
                    const double *params, int params_count, const double *kf_cov, double *state, double *xhat);

/* ---- the perturbed loop whose controller sees the observer's estimate instead of the raw measurement ------------- *
 * For k = 0 .. k_sim-1, in ONE launch:
 *   y_k = x_k + v_k
 *   xhat_k = ntm_kf_step(y_k, u_{k-1}; profile, params, kf_cov, its own record)   (fresh at k = 0: xhat_0 = y_0)
 *   u_k, U_k = one ntm_mpc_step_sc (NTM_STATE_ROWS_OFF: ntm_mpc_step) at xhat_k
 *   x_{k+1} = ntm_plant_step(x_k, u_k; plant_params, plant_profile) + d_k
 * bit for bit, up to and including the step at which a scenario turns infeasible.  Every other argument and output
 * means what it means in ntm_mpc_closed_loop_perturbed_sc: xk and cost are the true states, the offline build and the
 * frozen rows come from xhat_0 = y_0, the x_0 block of getWLc.m:30 tests xhat_k, and after an infeasible step the
 * scenario ends as there.  xhat: 2*k_sim doubles per scenario in `layout`, element 2k + i (or NULL): the estimate the
 * controller used at step k, NaN after an infeasible step.  kf_cov is required (the _perturbed entries are the loop
 * without an observer).  The filter records live in a handle-owned device buffer and every input travels with the
 * launch: the _dev entry queues one launch and no copy.
 * NTM_ERR_INVALID: whatever ntm_mpc_closed_loop_perturbed_sc or ntm_kf_step rejects. */
int ntm_mpc_closed_loop_observed(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                                 const double *x0, const double *params, int params_count, int state_rows,
                                 const double *xbounds, const double *plant_params, int plant_params_count,
                                 int plant_profile, const double *w, const double *v, const double *kf_cov,
                                 double *xhat, double *xk, double *uk, double *Uk, double *cost, int *inner_iters,
                                 int *qp_iters, int *status);
int ntm_mpc_closed_loop_observed_dev(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim,
                                     double eps, const double *x0, const double *params, int params_count,
                                     int state_rows, const double *xbounds, const double *plant_params,
                                     int plant_params_count, int plant_profile, const double *w, const double *v,
                                     const double *kf_cov, double *xhat, double *xk, double *uk, double *Uk,
                                     double *cost, int *inner_iters, int *qp_iters, int *status);

/* ---- the loop on EVERY visible GPU from ONE host process (what a MEX gateway can reach; SURVEY 8e) ------------- *
 * Replaces the same lines as ntm_mpc_closed_loop[_sc] (NTM_MPC_Sim.m:63-73,80-131); host pointers, same argument
 * meaning, no handle: the library keeps one pooled handle per device.  Scenarios never interact (:93-131 has no
 * cross-scenario term), so device g of n_devices owns the contiguous shard [g*ceil(S/n), min(S,(g+1)*ceil(S/n))) and
 * moves it straight between the caller's arrays and its own HBM on its own host thread and stream -- no collective,
 * the D2H copy of each shard IS the gather.  devices = NULL: ordinals 0..n_devices-1; n_devices = 0: every visible
 * device.  params_count is 1 or S.  state_rows / xbounds as in ntm_mpc_closed_loop_sc (NTM_STATE_ROWS_OFF, NULL for
 * the EC-power box only).  Results are bit-identical to the single-device call for every n_devices.  The pooled
 * handles are created on first use, before the arguments of that call are checked against each device. */
int ntm_device_count(int *count);
long long ntm_pool_launch_count(int device);   /* kernels launched so far by the pooled handle of `device`, -1 if none */
int ntm_mpc_closed_loop_multi(int n_devices, const int *devices, int layout, int profile, int S, int N, int k_sim,
                              int i_sim, double eps, const double *x0, const double *params, int params_count,
                              int state_rows, const double *xbounds, double *xk, double *uk, double *Uk, double *cost,
                              int *inner_iters, int *qp_iters, int *status);

/* ---- resident variant writing ONE packed record per scenario (multi-process callers gather it with a single
 * collective: SURVEY 8e "one ncclAllGather of per-scenario outputs") ------------------------------------------------ *
 * x0[2*S], params (scenario-slowest, NTM_LAYOUT_MATLAB) -> rec[NTM_REC_DOUBLES(k_sim)*S]:
 *   rec[s*ld + 0 .. 2(k_sim+1))  xk(:, 1:k_sim+1) column-major      (NTM_MPC_Sim.m:82)
 *   rec[s*ld + 2(k_sim+1) + k]   uk(k+1)                            (:83,107)
 *   rec[s*ld + 3 k_sim + 2]      cost,   rec[s*ld + 3 k_sim + 3]  status word as a double (0..3)
 * inner_iters / qp_iters [k_sim*S] may be NULL. */
#define NTM_REC_DOUBLES(k_sim) (3 * (k_sim) + 4)
int ntm_mpc_closed_loop_rec_dev(ntm_handle *h, int profile, int S, int N, int k_sim, int i_sim, double eps,
                                const double *x0, const double *params, int params_count, int state_rows,
                                const double *xbounds, double *rec, int *inner_iters, int *qp_iters);

/* ---- getWLc.m:1-63 (state + input constraint condensation; SURVEY 8f-1, defect D9 repaired) ----------- *
 * Phi[4N*S], Gamma[2N*N*S], Lambda[2N*S] + bounds -> W[(6N+4)*2*S], L[(6N+4)*N*S], c[(6N+4)*S] of
 * L*U <= c + W*x.  bounds = {xmax(1), xmax(2), xmin(1), xmin(2), umax, umin} on the HOST in both variants (six
 * scalars shared by all scenarios, like the script's xmax/xmin/umax/umin, NTM_MPC_Sim.m:44-50).                  */
int ntm_getWLc(ntm_handle *h, int layout, int S, int N, const double *bounds, const double *Gamma, const double *Phi,
               const double *Lambda, double *W, double *L, double *c);
int ntm_getWLc_dev(ntm_handle *h, int layout, int S, int N, const double *bounds, const double *Gamma,
                   const double *Phi, const double *Lambda, double *W, double *L, double *c);

/* ---- Monte-Carlo back end (SURVEY 8f-3): on-device reduction of a batch of closed-loop results ---------- *
 * Reads the outputs of ntm_mpc_closed_loop (xk[2*(k_sim+1)*S], uk[k_sim*S], cost[S], status[S], all in `layout`) and
 * the parameter block (umin/umax per scenario) and reduces them to NTM_MC_NSTAT doubles:
 *   [0] scenarios with status OK, [1] iteration-cap, [2] non-finite, [3] infeasible   (non-finite and infeasible ones are excluded below)
 *   [4] sum cost, [5] sum cost^2, [6] min cost, [7] max cost
 *   [8] sum w_final, [9] sum w_final^2, [10] min w_final, [11] max w_final      (w = island width, xk(1,end))
 *   [12] scenarios with w_final < w_suppressed, [13] sum of the first step index with w < w_suppressed, [14] their count
 *   [15] input samples at umin, [16] at umax, [17] all input samples, [18] sum of u      (active-bound fraction, mean power)
 *   [19] state samples (k >= 1) with w outside [xmin(1), xmax(1)], [20] omega outside [xmin(2), xmax(2)], [21] all state samples
 *   [22 .. 22+NTM_MC_NBINS) histogram of w_final over [0, hist_max) in equal bins (last bin takes everything above)
 * bounds = {xmin(1), xmax(1), xmin(2), xmax(2)} (NTM_MPC_Sim.m:44-45) on the HOST in both variants; `out` is a host
 * pointer (ntm_mc_stats) or a device pointer (ntm_mc_stats_dev).  Sums are order-dependent at rounding level. */
#define NTM_MC_NBINS 32
#define NTM_MC_NSTAT (22 + NTM_MC_NBINS)
int ntm_mc_stats(ntm_handle *h, int layout, int S, int k_sim, const double *xk, const double *uk, const double *cost,
                 const int *status, const double *params, int params_count, const double *bounds,
                 double w_suppressed, double hist_max, double *out);
int ntm_mc_stats_dev(ntm_handle *h, int layout, int S, int k_sim, const double *xk, const double *uk,
                     const double *cost, const int *status, const double *params, int params_count,
                     const double *bounds, double w_suppressed, double hist_max, double *out);

/* the same reduction with the EC-power box as two compact device arrays umin[S], umax[S] (bounds_count = S) or one shared
 * pair (bounds_count = 1) instead of the parameter block: in the MATLAB layout the block costs a 128-byte line per
 * scenario for these two doubles. */
int ntm_mc_stats_ub_dev(ntm_handle *h, int layout, int S, int k_sim, const double *xk, const double *uk,
                        const double *cost, const int *status, const double *umin, const double *umax, int bounds_count,
                        const double *bounds, double w_suppressed, double hist_max, double *out);

/* ---- measurement aid: register-resident DFMA chain, returns achieved FP64 TFLOP/s ------------ */
int ntm_fp64_peak(ntm_handle *h, int iters, double *tflops_dfma, double *ms);
/* the same for the FP64 tensor cores: register-resident mma.sync.m8n8k4.f64 (DMMA.8x8x4) chains */
int ntm_dmma_peak(ntm_handle *h, int iters, double *tflops_dmma, double *ms);

#ifdef __cplusplus
}
#endif
#endif /* NTM_MPC_H */
