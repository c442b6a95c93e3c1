/* ntm_mex.c -- MATLAB/Octave MEX gateways over the C ABI of include/ntm_mpc.h.
 *
 * One source, one gateway per reference function: compile with -DNTM_MEX_FN=<id>, name the output after the
 * reference file it shadows (a rho1.mexa64 next to rho1.m wins over the .m on the MATLAB path):
 *
 *   id  output name              replaces                      call forms accepted
 *   1   rho1                     rho1.m:1-3                    rho1(x)            rho1(x, wmarg)
 *   2   rho2                     rho2.m:1-3                    rho2(x)
 *   3   rho3                     rho3.m:1-4                    rho3(x)            rho3(x, w_dep)
 *   4   A                        A.m:1-3                       A(r1, r2)          A(r1,r2,kappa,taur,Ts,zeta,rs,a,TE)
 *   5   B                        B.m:1-3                       B(r3)              B(r3,wdep,kappa,Ts,etaCD)
 *   6   Rho_to_PhiGammaLambda    Rho_to_PhiGammaLambda.m:1-54  (Rho1,Rho2,Rho3)   (Rho1,Rho2,Rho3,A,B,C)
 *   7   ntm_qp_box               quadprog call NTM_MPC_Sim.m:97 [U,exitflag,iters] = ntm_qp_box(G,F,lb,ub)
 *   8   ntm_mpc_batch            loop NTM_MPC_Sim.m:93-131      [xk,uk,cost,inner,status] = ntm_mpc_batch(x0,params,N,k_sim,i_sim,eps,profile[,state_rows,xmin,xmax])
 *   9   getWLc                   getWLc.m:1-63                 [W,L,c] = getWLc(xmax,xmin,umax,umin,Gamma,Phi,Lambda)
 *   10  quadprog                 quadprog call NTM_MPC_Sim.m:97 [U,fval,exitflag] = quadprog(H,f,A,b,[],[],lb,ub,x0,options)
 *                                (shadows the Optimization Toolbox function: input-box rows become bounds, state rows stay)
 *   11  ntm_mpc_step             one step NTM_MPC_Sim.m:94-128  [u,state,U,inner,status] = ntm_mpc_step(state,x,params,N,i_sim,eps,profile[,state_rows,xmin,xmax])
 *                                (no plant: the script's `for k` loop keeps its own plant code and passes state back in)
 *   12  ntm_mpc_batch_perturbed  the loop vs a perturbed plant  [xk,uk,cost,inner,status] = ntm_mpc_batch_perturbed(x0,params,N,k_sim,i_sim,eps,profile,plant_params,plant_profile,w,v)
 *
 * The short forms are the ones NTM_MPC_Sim.m actually uses (:63-66,:113-119,:130); the missing trailing arguments
 * are fetched from the caller's workspace under the script's own variable names (kappa :24, tau_r :9, Ts :31,
 * zeta :25, rs :10, a :11, tau_E :14, w_dep :6, eta_CD :12, w_marg :7, C :37).  x may be 2x1 or 2xS (columns are
 * scenarios); rho vectors may be rows or columns (N = numel, repair of defect D4); B is returned as the 2x1 column
 * the script needs (defect D7).  All data are real doubles, column-major, passed straight to the MATLAB-layout
 * entry points.  Every CUDA resource is owned by a static handle (mexLock + mexAtExit), and errors are raised with
 * mexErrMsgIdAndTxt only after the C ABI call has returned (nothing to unwind).  There is no CPU fallback.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "mex.h"
#include "ntm_mpc.h"

#ifndef NTM_MEX_FN
#error "compile with -DNTM_MEX_FN=<1..12>"
#endif

static ntm_handle *g_h = NULL;

static void cleanup(void) {
    if (g_h) { ntm_destroy(g_h); g_h = NULL; }
}

static ntm_handle *handle(void) {
    if (!g_h) {
        if (ntm_create(&g_h, 0) != NTM_OK) mexErrMsgIdAndTxt("ntm:cuda", ntm_last_error());
        mexLock();
        mexAtExit(cleanup);
    }
    return g_h;
}

static void check(int rc) {
    if (rc != NTM_OK) mexErrMsgIdAndTxt("ntm:call", ntm_last_error());
}

static int is_real_double(const mxArray *a) { return a && mxIsDouble(a) && !mxIsComplex(a); }

static double scalar_arg(int nrhs, const mxArray *prhs[], int pos, const char *ws_name) {
    if (pos < nrhs) {
        if (!is_real_double(prhs[pos]) || mxGetNumberOfElements(prhs[pos]) != 1)
            mexErrMsgIdAndTxt("ntm:arg", "scalar real double expected");
        return mxGetScalar(prhs[pos]);
    }
    {
        const mxArray *v = mexGetVariablePtr("caller", ws_name);
        if (!is_real_double(v) || mxGetNumberOfElements(v) != 1) {
            mexErrMsgIdAndTxt("ntm:workspace", "Not enough input arguments and the caller workspace does not define the missing constant.");
            return 0.0;
        }
        return mxGetScalar(v);
    }
}

static void blank_params(double *p) {
    memset(p, 0, sizeof(double) * NTM_NPARAM);
    p[7] = 1.0;            /* w_dep: keeps the unused rho3 finite */
    p[12] = p[14] = 1.0;   /* Q = I */
}

/* hoisted coefficients in the evaluation order of A.m:2 / B.m:2 */
static void model_params(double *p, double kappa, double taur, double Ts, double zeta, double rs, double a, double TE,
                         double wdep, double etaCD) {
    blank_params(p);
    p[0] = (4.0 / 3.0) * (kappa * rs / (0.82 * taur)) * Ts;
    p[1] = Ts / (zeta * (a * a * a));
    p[2] = 1 - Ts / TE;
    p[3] = (kappa * Ts * etaCD / wdep);
    p[7] = wdep;
}

static int states_arg(const mxArray *x) {
    if (is_real_double(x) && mxGetM(x) == 1 && mxGetN(x) == 2) return 1;     /* a single state given as a row: x(1), x(2) */
    if (!is_real_double(x) || mxGetM(x) != 2) mexErrMsgIdAndTxt("ntm:arg", "x must be a real 2 x S matrix ([w; omega] per column)");
    return (int)mxGetN(x);
}

void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    double prm[NTM_NPARAM];
    (void)nlhs;
#if NTM_MEX_FN == 1 || NTM_MEX_FN == 2 || NTM_MEX_FN == 3
    {
        int S, profile = 0;
        mxArray *r1, *r2, *r3;
        if (nrhs < 1 || nrhs > 2) mexErrMsgIdAndTxt("ntm:arg", "usage: rho(x) or rho(x, constant)");
        S = states_arg(prhs[0]);
        blank_params(prm);
#if NTM_MEX_FN == 1
        { double wm = scalar_arg(nrhs, prhs, 1, "w_marg"); prm[6] = wm * wm; }
        if (mexGetVariablePtr("caller", "ntm_rho1_sq")) profile |= NTM_PROFILE_RHO1_SQ;
#elif NTM_MEX_FN == 3
        prm[7] = scalar_arg(nrhs, prhs, 1, "w_dep");
#endif
        r1 = mxCreateDoubleMatrix(1, S, mxREAL); r2 = mxCreateDoubleMatrix(1, S, mxREAL); r3 = mxCreateDoubleMatrix(1, S, mxREAL);
        check(ntm_rho(handle(), NTM_LAYOUT_MATLAB, profile, S, mxGetPr(prhs[0]), prm, 1, mxGetPr(r1), mxGetPr(r2), mxGetPr(r3)));
#if NTM_MEX_FN == 1
        plhs[0] = r1; mxDestroyArray(r2); mxDestroyArray(r3);
#elif NTM_MEX_FN == 2
        plhs[0] = r2; mxDestroyArray(r1); mxDestroyArray(r3);
#else
        plhs[0] = r3; mxDestroyArray(r1); mxDestroyArray(r2);
#endif
    }
#elif NTM_MEX_FN == 4
    {   /* A(rho1, rho2 [, kappa, taur, Ts, zeta, rs, a, TE]) */
        int S, i;
        mxArray *Aout, *Bout, *zero;
        if (nrhs != 2 && nrhs != 9) mexErrMsgIdAndTxt("ntm:arg", "usage: A(rho1, rho2) or A(rho1, rho2, kappa, taur, Ts, zeta, rs, a, TE)");
        if (!is_real_double(prhs[0]) || !is_real_double(prhs[1]) ||
            mxGetNumberOfElements(prhs[0]) != mxGetNumberOfElements(prhs[1]))
            mexErrMsgIdAndTxt("ntm:arg", "rho1 and rho2 must be real doubles of equal size");
        S = (int)mxGetNumberOfElements(prhs[0]);
        model_params(prm, scalar_arg(nrhs, prhs, 2, "kappa"), scalar_arg(nrhs, prhs, 3, "tau_r"), scalar_arg(nrhs, prhs, 4, "Ts"),
                     scalar_arg(nrhs, prhs, 5, "zeta"), scalar_arg(nrhs, prhs, 6, "rs"), scalar_arg(nrhs, prhs, 7, "a"),
                     scalar_arg(nrhs, prhs, 8, "tau_E"), 1.0, 0.0);
        Aout = (S == 1) ? mxCreateDoubleMatrix(2, 2, mxREAL) : mxCreateDoubleMatrix(4, S, mxREAL);
        Bout = mxCreateDoubleMatrix(2, S, mxREAL);
        zero = mxCreateDoubleMatrix(1, S, mxREAL);
        for (i = 0; i < S; ++i) mxGetPr(zero)[i] = 0.0;
        check(ntm_lpv_AB(handle(), NTM_LAYOUT_MATLAB, S, mxGetPr(prhs[0]), mxGetPr(prhs[1]), mxGetPr(zero), prm, 1, mxGetPr(Aout), mxGetPr(Bout)));
        plhs[0] = Aout; mxDestroyArray(Bout); mxDestroyArray(zero);
    }
#elif NTM_MEX_FN == 5
    {   /* B(rho3 [, wdep, kappa, Ts, etaCD]) */
        int S, i;
        mxArray *Aout, *Bout, *zero;
        if (nrhs != 1 && nrhs != 5) mexErrMsgIdAndTxt("ntm:arg", "usage: B(rho3) or B(rho3, wdep, kappa, Ts, etaCD)");
        if (!is_real_double(prhs[0])) mexErrMsgIdAndTxt("ntm:arg", "rho3 must be a real double");
        S = (int)mxGetNumberOfElements(prhs[0]);
        {
            double wdep = scalar_arg(nrhs, prhs, 1, "w_dep"), kappa = scalar_arg(nrhs, prhs, 2, "kappa");
            double Ts = scalar_arg(nrhs, prhs, 3, "Ts"), eta = scalar_arg(nrhs, prhs, 4, "eta_CD");
            model_params(prm, kappa, 1.0, Ts, 1.0, 1.0, 1.0, 1.0, wdep, eta);
        }
        Aout = mxCreateDoubleMatrix(4, S, mxREAL); Bout = mxCreateDoubleMatrix(2, S, mxREAL);
        zero = mxCreateDoubleMatrix(1, S, mxREAL);
        for (i = 0; i < S; ++i) mxGetPr(zero)[i] = 0.0;
        check(ntm_lpv_AB(handle(), NTM_LAYOUT_MATLAB, S, mxGetPr(zero), mxGetPr(zero), mxGetPr(prhs[0]), prm, 1, mxGetPr(Aout), mxGetPr(Bout)));
        plhs[0] = Bout; mxDestroyArray(Aout); mxDestroyArray(zero);
    }
#elif NTM_MEX_FN == 6
    {   /* [Phi, Gamma, Lambda] = Rho_to_PhiGammaLambda(Rho1, Rho2, Rho3 [, A, B, C]) */
        int N, profile = 0;
        const mxArray *Cv;
        mxArray *Phi, *Gam, *Lam;
        if (nrhs != 3 && nrhs != 6) mexErrMsgIdAndTxt("ntm:arg", "usage: Rho_to_PhiGammaLambda(Rho1,Rho2,Rho3) or (Rho1,Rho2,Rho3,A,B,C)");
        if (!is_real_double(prhs[0]) || !is_real_double(prhs[1]) || !is_real_double(prhs[2]))
            mexErrMsgIdAndTxt("ntm:arg", "Rho1..3 must be real double vectors");
        N = (int)mxGetNumberOfElements(prhs[0]);                       /* numel: rows or columns (D4) */
        if (N < 1 || N > NTM_MAX_HORIZON || (int)mxGetNumberOfElements(prhs[1]) != N || (int)mxGetNumberOfElements(prhs[2]) != N)
            mexErrMsgIdAndTxt("ntm:arg", "Rho1..3 must have the same length 1..128");
        /* the A/B handles of the 6-argument form cannot run on the GPU: the constants they close over are read from
           the caller workspace, exactly as for the 3-argument form the script uses */
        model_params(prm, scalar_arg(0, prhs, 0, "kappa"), scalar_arg(0, prhs, 0, "tau_r"), scalar_arg(0, prhs, 0, "Ts"),
                     scalar_arg(0, prhs, 0, "zeta"), scalar_arg(0, prhs, 0, "rs"), scalar_arg(0, prhs, 0, "a"),
                     scalar_arg(0, prhs, 0, "tau_E"), scalar_arg(0, prhs, 0, "w_dep"), scalar_arg(0, prhs, 0, "eta_CD"));
        Cv = (nrhs == 6) ? prhs[5] : mexGetVariablePtr("caller", "C");
        if (!is_real_double(Cv) || mxGetNumberOfElements(Cv) != 2) mexErrMsgIdAndTxt("ntm:arg", "C must be a real 2-vector");
        prm[4] = mxGetPr(Cv)[0]; prm[5] = mxGetPr(Cv)[1];
        if (mexGetVariablePtr("caller", "ntm_gamma_index_i")) profile |= NTM_PROFILE_GAMMA_I;
        Phi = mxCreateDoubleMatrix(2 * N, 2, mxREAL); Gam = mxCreateDoubleMatrix(2 * N, N, mxREAL); Lam = mxCreateDoubleMatrix(2 * N, 1, mxREAL);
        check(ntm_condense(handle(), NTM_LAYOUT_MATLAB, profile, 1, N, mxGetPr(prhs[0]), mxGetPr(prhs[1]), mxGetPr(prhs[2]), prm, 1,
                           mxGetPr(Phi), mxGetPr(Gam), mxGetPr(Lam)));
        plhs[0] = Phi;
        if (nlhs > 1) plhs[1] = Gam; else mxDestroyArray(Gam);
        if (nlhs > 2) plhs[2] = Lam; else mxDestroyArray(Lam);
    }
#elif NTM_MEX_FN == 7
    {   /* [U, exitflag, iters] = ntm_qp_box(G, F, lb, ub) -- exitflag as quadprog: 1 solved, 0 iteration cap, -3 non-finite */
        int N, i, it = 0, st = 0;
        mxArray *U, *lb, *ub;
        if (nrhs != 4) mexErrMsgIdAndTxt("ntm:arg", "usage: [U, exitflag, iters] = ntm_qp_box(G, F, lb, ub)");
        for (i = 0; i < 4; ++i) if (!is_real_double(prhs[i])) mexErrMsgIdAndTxt("ntm:arg", "real double inputs expected");
        N = (int)mxGetM(prhs[0]);
        if (N < 1 || N > NTM_MAX_HORIZON || (int)mxGetN(prhs[0]) != N || (int)mxGetNumberOfElements(prhs[1]) != N)
            mexErrMsgIdAndTxt("ntm:arg", "G must be N x N and F of length N, 1 <= N <= 128");
        lb = mxCreateDoubleMatrix(N, 1, mxREAL); ub = mxCreateDoubleMatrix(N, 1, mxREAL);
        for (i = 0; i < N; ++i) {
            mxGetPr(lb)[i] = mxGetPr(prhs[2])[mxGetNumberOfElements(prhs[2]) == 1 ? 0 : i];
            mxGetPr(ub)[i] = mxGetPr(prhs[3])[mxGetNumberOfElements(prhs[3]) == 1 ? 0 : i];
        }
        U = mxCreateDoubleMatrix(N, 1, mxREAL);
        check(ntm_qp_box(handle(), NTM_LAYOUT_MATLAB, 1, N, mxGetPr(prhs[0]), mxGetPr(prhs[1]), mxGetPr(lb), mxGetPr(ub), 1, mxGetPr(U), &it, &st));
        mxDestroyArray(lb); mxDestroyArray(ub);
        plhs[0] = U;
        if (nlhs > 1) plhs[1] = mxCreateDoubleScalar(st == NTM_SCN_OK ? 1.0 : (st == NTM_SCN_QP_ITER_CAP ? 0.0 : -3.0));
        if (nlhs > 2) plhs[2] = mxCreateDoubleScalar((double)it);
    }
#elif NTM_MEX_FN == 8
    {   /* [xk, uk, cost, inner, status] = ntm_mpc_batch(x0 (2xS), params (16x1 | 16xS), N, k_sim, i_sim, eps, profile
         *                                                  [, state_rows, xmin (2x1), xmax (2x1)])
         * state_rows: 0 box QP, 1 getWLc's state rows rebuilt at every re-condensation, 2 frozen at the offline build
         * as NTM_MPC_Sim.m:74 does; xmin / xmax as NTM_MPC_Sim.m:44-45 */
        int S, N, k_sim, i_sim, profile, pc, i, srows = 0;
        double eps, xb[4] = {0.0, 0.0, 0.0, 0.0};
        mxArray *xk, *uk, *cost, *inner, *status;
        int *ibuf;
        if (nrhs != 7 && nrhs != 10)
            mexErrMsgIdAndTxt("ntm:arg", "usage: [xk,uk,cost,inner,status] = ntm_mpc_batch(x0, params, N, k_sim, i_sim, eps, profile [, state_rows, xmin, xmax])");
        if (nrhs == 10) {
            srows = (int)scalar_arg(nrhs, prhs, 7, "");
            if (!is_real_double(prhs[8]) || !is_real_double(prhs[9]) || mxGetNumberOfElements(prhs[8]) != 2 ||
                mxGetNumberOfElements(prhs[9]) != 2)
                mexErrMsgIdAndTxt("ntm:arg", "xmin and xmax must be real double 2-vectors");
            xb[0] = mxGetPr(prhs[8])[0]; xb[1] = mxGetPr(prhs[9])[0]; xb[2] = mxGetPr(prhs[8])[1]; xb[3] = mxGetPr(prhs[9])[1];
        }
        S = states_arg(prhs[0]);
        if (!is_real_double(prhs[1]) || mxGetM(prhs[1]) != NTM_NPARAM || ((int)mxGetN(prhs[1]) != 1 && (int)mxGetN(prhs[1]) != S))
            mexErrMsgIdAndTxt("ntm:arg", "params must be 16 x 1 or 16 x S (see ntm_mpc.h)");
        pc = (int)mxGetN(prhs[1]);
        N = (int)scalar_arg(nrhs, prhs, 2, ""); k_sim = (int)scalar_arg(nrhs, prhs, 3, ""); i_sim = (int)scalar_arg(nrhs, prhs, 4, "");
        eps = scalar_arg(nrhs, prhs, 5, ""); profile = (int)scalar_arg(nrhs, prhs, 6, "");
        if (N < 1 || N > NTM_MAX_HORIZON || k_sim < 0 || i_sim < 1) mexErrMsgIdAndTxt("ntm:arg", "N in 1..128, k_sim >= 0, i_sim >= 1");
        xk = mxCreateDoubleMatrix(2 * (k_sim + 1), S, mxREAL); uk = mxCreateDoubleMatrix(k_sim, S, mxREAL);
        cost = mxCreateDoubleMatrix(1, S, mxREAL); inner = mxCreateDoubleMatrix(k_sim, S, mxREAL); status = mxCreateDoubleMatrix(1, S, mxREAL);
        ibuf = (int *)mxMalloc(sizeof(int) * ((size_t)k_sim * S + S + 1));
        {   /* Every visible GPU from this one interpreter process: contiguous scenario shards, >= NTM_MEX_MIN_SHARD (default
             * 1024) scenarios per device, at most NTM_MEX_DEVICES devices (default: all).  One device: the plain entry. */
            int ndev = 1, use, min_shard = 1024;
            const char *ev = getenv("NTM_MEX_DEVICES"), *ms = getenv("NTM_MEX_MIN_SHARD");
            if (ntm_device_count(&ndev) != NTM_OK) ndev = 1;
            if (ev && atoi(ev) > 0 && atoi(ev) < ndev) ndev = atoi(ev);
            if (ms && atoi(ms) > 0) min_shard = atoi(ms);
            use = S / min_shard < ndev ? S / min_shard : ndev;
            if (use >= 2)
                check(ntm_mpc_closed_loop_multi(use, NULL, NTM_LAYOUT_MATLAB, profile, S, N, k_sim, i_sim, eps, mxGetPr(prhs[0]),
                                                mxGetPr(prhs[1]), pc, srows, xb, mxGetPr(xk), mxGetPr(uk), NULL, mxGetPr(cost), ibuf,
                                                NULL, ibuf + (size_t)k_sim * S));
            else
                check(ntm_mpc_closed_loop_sc(handle(), NTM_LAYOUT_MATLAB, profile, S, N, k_sim, i_sim, eps, mxGetPr(prhs[0]), mxGetPr(prhs[1]), pc,
                                             srows, xb, mxGetPr(xk), mxGetPr(uk), NULL, mxGetPr(cost), ibuf, NULL, ibuf + (size_t)k_sim * S));
        }
        for (i = 0; i < k_sim * S; ++i) mxGetPr(inner)[i] = (double)ibuf[i];
        for (i = 0; i < S; ++i) mxGetPr(status)[i] = (double)ibuf[(size_t)k_sim * S + i];
        mxFree(ibuf);
        plhs[0] = xk;
        if (nlhs > 1) plhs[1] = uk; else mxDestroyArray(uk);
        if (nlhs > 2) plhs[2] = cost; else mxDestroyArray(cost);
        if (nlhs > 3) plhs[3] = inner; else mxDestroyArray(inner);
        if (nlhs > 4) plhs[4] = status; else mxDestroyArray(status);
    }
#elif NTM_MEX_FN == 9
    {   /* [W, L, c] = getWLc(xmax, xmin, umax, umin, Gamma, Phi, Lambda)  -- getWLc.m:1 */
        int N, R, i;
        double b[6];
        mxArray *W, *L, *c;
        if (nrhs != 7) mexErrMsgIdAndTxt("ntm:arg", "usage: [W, L, c] = getWLc(xmax, xmin, umax, umin, Gamma, Phi, Lambda)");
        for (i = 0; i < 7; ++i) if (!is_real_double(prhs[i])) mexErrMsgIdAndTxt("ntm:arg", "real double inputs expected");
        if (mxGetNumberOfElements(prhs[0]) != 2 || mxGetNumberOfElements(prhs[1]) != 2 || mxGetNumberOfElements(prhs[2]) != 1 ||
            mxGetNumberOfElements(prhs[3]) != 1)
            mexErrMsgIdAndTxt("ntm:arg", "xmax, xmin must have 2 entries and umax, umin 1 (nx = 2, nu = 1)");
        N = (int)mxGetN(prhs[4]);
        if (N < 1 || N > NTM_MAX_HORIZON || (int)mxGetM(prhs[4]) != 2 * N || (int)mxGetM(prhs[5]) != 2 * N || (int)mxGetN(prhs[5]) != 2 ||
            (int)mxGetNumberOfElements(prhs[6]) != 2 * N)
            mexErrMsgIdAndTxt("ntm:arg", "Gamma must be 2N x N, Phi 2N x 2, Lambda 2N x 1, 1 <= N <= 128");
        b[0] = mxGetPr(prhs[0])[0]; b[1] = mxGetPr(prhs[0])[1]; b[2] = mxGetPr(prhs[1])[0]; b[3] = mxGetPr(prhs[1])[1];
        b[4] = mxGetScalar(prhs[2]); b[5] = mxGetScalar(prhs[3]);
        R = 6 * N + 4;
        W = mxCreateDoubleMatrix(R, 2, mxREAL); L = mxCreateDoubleMatrix(R, N, mxREAL); c = mxCreateDoubleMatrix(R, 1, mxREAL);
        check(ntm_getWLc(handle(), NTM_LAYOUT_MATLAB, 1, N, b, mxGetPr(prhs[4]), mxGetPr(prhs[5]), mxGetPr(prhs[6]), mxGetPr(W), mxGetPr(L), mxGetPr(c)));
        plhs[0] = W;
        if (nlhs > 1) plhs[1] = L; else mxDestroyArray(L);
        if (nlhs > 2) plhs[2] = c; else mxDestroyArray(c);
    }
#elif NTM_MEX_FN == 10
    {   /* [U, fval, exitflag] = quadprog(H, f, A, b, Aeq, beq, lb, ub, x0, options) -- the call of NTM_MPC_Sim.m:97 as written.
         * Rows of A are split here: one non-zero -> a bound (getWLc.m:14-23), none -> feasibility of b (the x_0 block,
         * getWLc.m:30, defect D18), the rest -> general rows for ntm_qp_ineq.  exitflag 1 / 0 / -2 / -3. */
        int N, M = 0, Mg = 0, i, j, it = 0, st = 0, feasible = 1;
        const double *H, *f, *A = NULL, *b = NULL;
        double *lb, *ub, *Lg = NULL, *bg = NULL, fval = 0.0;
        int *gen = NULL;
        mxArray *U;
        if (nrhs < 2) mexErrMsgIdAndTxt("ntm:arg", "usage: [U, fval, exitflag] = quadprog(H, f, A, b, [], [], lb, ub)");
        for (i = 0; i < nrhs && i < 8; ++i)
            if (mxGetNumberOfElements(prhs[i]) && !is_real_double(prhs[i])) mexErrMsgIdAndTxt("ntm:arg", "real double inputs expected");
        N = (int)mxGetM(prhs[0]);
        if (N < 1 || N > NTM_MAX_HORIZON || (int)mxGetN(prhs[0]) != N || (int)mxGetNumberOfElements(prhs[1]) != N)
            mexErrMsgIdAndTxt("ntm:arg", "H must be N x N and f of length N, 1 <= N <= 128");
        if ((nrhs > 4 && mxGetNumberOfElements(prhs[4])) || (nrhs > 5 && mxGetNumberOfElements(prhs[5])))
            mexErrMsgIdAndTxt("ntm:arg", "equality constraints are not supported (NTM_MPC_Sim.m:97 passes [] for Aeq, beq)");
        H = mxGetPr(prhs[0]); f = mxGetPr(prhs[1]);
        if (nrhs > 3 && mxGetNumberOfElements(prhs[2])) {
            M = (int)mxGetM(prhs[2]);
            if ((int)mxGetN(prhs[2]) != N || (int)mxGetNumberOfElements(prhs[3]) != M)
                mexErrMsgIdAndTxt("ntm:arg", "A must be M x N and b of length M");
            A = mxGetPr(prhs[2]); b = mxGetPr(prhs[3]);
        }
        lb = (double *)mxMalloc(sizeof(double) * 2 * (size_t)N); ub = lb + N;
        for (j = 0; j < N; ++j) { lb[j] = -HUGE_VAL; ub[j] = HUGE_VAL; }
        if (nrhs > 6 && mxGetNumberOfElements(prhs[6])) {
            if ((int)mxGetNumberOfElements(prhs[6]) != N) mexErrMsgIdAndTxt("ntm:arg", "lb must have N entries");
            for (j = 0; j < N; ++j) lb[j] = mxGetPr(prhs[6])[j];
        }
        if (nrhs > 7 && mxGetNumberOfElements(prhs[7])) {
            if ((int)mxGetNumberOfElements(prhs[7]) != N) mexErrMsgIdAndTxt("ntm:arg", "ub must have N entries");
            for (j = 0; j < N; ++j) ub[j] = mxGetPr(prhs[7])[j];
        }
        gen = (int *)mxMalloc(sizeof(int) * (size_t)(M + 1));
        for (i = 0; i < M; ++i) {
            int nnz = 0, col = -1;
            for (j = 0; j < N; ++j) if (A[i + (size_t)M * j] != 0.0) { ++nnz; col = j; }
            if (nnz == 0) { if (b[i] < 0.0) feasible = 0; }
            else if (nnz == 1) {
                const double a = A[i + (size_t)M * col], v = b[i] / a;
                if (a > 0.0) { if (v < ub[col]) ub[col] = v; } else { if (v > lb[col]) lb[col] = v; }
            } else gen[Mg++] = i;
        }
        for (j = 0; j < N; ++j) {
            if (!(lb[j] > -HUGE_VAL) || !(ub[j] < HUGE_VAL))
                mexErrMsgIdAndTxt("ntm:arg", "every variable needs finite lower and upper bounds (getWLc.m:14-23 provides them)");
            if (lb[j] > ub[j]) { feasible = 0; ub[j] = lb[j]; }
        }
        U = mxCreateDoubleMatrix(N, 1, mxREAL);
        if (Mg > 0 && feasible) {
            Lg = (double *)mxMalloc(sizeof(double) * (size_t)Mg * (N + 1)); bg = Lg + (size_t)Mg * N;
            for (i = 0; i < Mg; ++i) {
                bg[i] = b[gen[i]];
                for (j = 0; j < N; ++j) Lg[i + (size_t)Mg * j] = A[gen[i] + (size_t)M * j];
            }
            check(ntm_qp_ineq(handle(), NTM_LAYOUT_MATLAB, 1, N, Mg, H, f, lb, ub, 1, Lg, bg, mxGetPr(U), &it, &st));
            mxFree(Lg);
        } else {
            check(ntm_qp_box(handle(), NTM_LAYOUT_MATLAB, 1, N, H, f, lb, ub, 1, mxGetPr(U), &it, &st));
        }
        if (!feasible) st = NTM_SCN_INFEASIBLE;
        for (i = 0; i < N; ++i) {
            double hu = 0.0;
            for (j = 0; j < N; ++j) hu += H[i + (size_t)N * j] * mxGetPr(U)[j];
            fval += mxGetPr(U)[i] * (0.5 * hu + f[i]);
        }
        mxFree(gen); mxFree(lb);
        plhs[0] = U;
        if (nlhs > 1) plhs[1] = mxCreateDoubleScalar(fval);
        if (nlhs > 2) plhs[2] = mxCreateDoubleScalar(st == NTM_SCN_OK ? 1.0 : (st == NTM_SCN_QP_ITER_CAP ? 0.0 : (st == NTM_SCN_INFEASIBLE ? -2.0 : -3.0)));
    }
#elif NTM_MEX_FN == 11
    {   /* [u, state, U, inner, status] = ntm_mpc_step(state, x (2xS), params (16x1 | 16xS), N, i_sim, eps, profile
         *                                              [, state_rows, xmin (2x1), xmax (2x1)])
         * One receding-horizon step at the measured states x; state = [] starts S fresh controllers, otherwise it is the
         * NTM_CTRL_DOUBLES(N) x S record this gateway returned last time (zeroing a column restarts that scenario).
         * state_rows / xmin / xmax as in ntm_mpc_batch (ntm_mpc_step_sc): an infeasible QP returns NaN u and U, status 3
         * and the record as it was.  Pass the same N, params, profile, state_rows and bounds on every call for the same
         * state. */
        int S, N, i_sim, profile, pc, i, srows = 0;
        double eps, xb[4] = {0.0, 0.0, 0.0, 0.0};
        size_t ld;
        mxArray *u, *st, *U, *inner, *status;
        int *ibuf;
        if (nrhs != 7 && nrhs != 10)
            mexErrMsgIdAndTxt("ntm:arg", "usage: [u, state, U, inner, status] = ntm_mpc_step(state, x, params, N, i_sim, eps, profile [, state_rows, xmin, xmax])");
        if (nrhs == 10) {
            srows = (int)scalar_arg(nrhs, prhs, 7, "");
            if (srows < 0 || srows > 2) mexErrMsgIdAndTxt("ntm:arg", "state_rows must be 0, 1 or 2");
            if (!is_real_double(prhs[8]) || !is_real_double(prhs[9]) || mxGetNumberOfElements(prhs[8]) != 2 ||
                mxGetNumberOfElements(prhs[9]) != 2)
                mexErrMsgIdAndTxt("ntm:arg", "xmin and xmax must be real double 2-vectors");
            xb[0] = mxGetPr(prhs[8])[0]; xb[1] = mxGetPr(prhs[9])[0]; xb[2] = mxGetPr(prhs[8])[1]; xb[3] = mxGetPr(prhs[9])[1];
            if (!(xb[0] <= xb[1] && xb[2] <= xb[3])) mexErrMsgIdAndTxt("ntm:arg", "xmin must be <= xmax");
        }
        S = states_arg(prhs[1]);
        if (!is_real_double(prhs[2]) || mxGetM(prhs[2]) != NTM_NPARAM || ((int)mxGetN(prhs[2]) != 1 && (int)mxGetN(prhs[2]) != S))
            mexErrMsgIdAndTxt("ntm:arg", "params must be 16 x 1 or 16 x S (see ntm_mpc.h)");
        pc = (int)mxGetN(prhs[2]);
        N = (int)scalar_arg(nrhs, prhs, 3, ""); i_sim = (int)scalar_arg(nrhs, prhs, 4, "");
        eps = scalar_arg(nrhs, prhs, 5, ""); profile = (int)scalar_arg(nrhs, prhs, 6, "");
        if (N < 1 || N > NTM_MAX_HORIZON || i_sim < 1) mexErrMsgIdAndTxt("ntm:arg", "N in 1..128, i_sim >= 1");
        if (profile & NTM_PROFILE_TAUE_W) mexErrMsgIdAndTxt("ntm:arg", "NTM_PROFILE_TAUE_W (128) is not supported by ntm_mpc_step");
        if (srows != 0 && (profile & (NTM_PROFILE_GAMMA_I | NTM_PROFILE_DENSE_G)) && N > 32)
            mexErrMsgIdAndTxt("ntm:arg", "state rows with NTM_PROFILE_GAMMA_I / DENSE_G need N <= 32");
        ld = (size_t)NTM_CTRL_DOUBLES(N);
        if (!is_real_double(prhs[0]))
            mexErrMsgIdAndTxt("ntm:arg", "state must be [] or a real double matrix");
        if (mxGetNumberOfElements(prhs[0]) != 0 && ((size_t)mxGetM(prhs[0]) != ld || (int)mxGetN(prhs[0]) != S))
            mexErrMsgIdAndTxt("ntm:arg", "state must be [] or NTM_CTRL_DOUBLES(N) = 7N+7 rows by S columns");
        st = mxCreateDoubleMatrix(ld, S, mxREAL);                  /* zeros: a fresh controller */
        if (mxGetNumberOfElements(prhs[0]) != 0) memcpy(mxGetPr(st), mxGetPr(prhs[0]), sizeof(double) * ld * (size_t)S);
        u = mxCreateDoubleMatrix(1, S, mxREAL); U = mxCreateDoubleMatrix(N, S, mxREAL);
        inner = mxCreateDoubleMatrix(1, S, mxREAL); status = mxCreateDoubleMatrix(1, S, mxREAL);
        ibuf = (int *)mxMalloc(sizeof(int) * (2 * (size_t)S + 1));
        check(ntm_mpc_step_sc(handle(), NTM_LAYOUT_MATLAB, profile, S, N, i_sim, eps, mxGetPr(prhs[1]), mxGetPr(prhs[2]), pc,
                              srows, xb, mxGetPr(st), mxGetPr(u), mxGetPr(U), ibuf, NULL, ibuf + S));
        for (i = 0; i < S; ++i) { mxGetPr(inner)[i] = (double)ibuf[i]; mxGetPr(status)[i] = (double)ibuf[S + i]; }
        mxFree(ibuf);
        plhs[0] = u;
        if (nlhs > 1) plhs[1] = st; else mxDestroyArray(st);
        if (nlhs > 2) plhs[2] = U; else mxDestroyArray(U);
        if (nlhs > 3) plhs[3] = inner; else mxDestroyArray(inner);
        if (nlhs > 4) plhs[4] = status; else mxDestroyArray(status);
    }
#elif NTM_MEX_FN == 12
    {   /* [xk, uk, cost, inner, status] = ntm_mpc_batch_perturbed(x0 (2xS), params (16x1 | 16xS), N, k_sim, i_sim, eps,
         *                                                           profile, plant_params, plant_profile, w, v)
         * The fused loop against a perturbed plant (ntm_mpc_closed_loop_perturbed), one device: the controller of
         * ntm_mpc_batch sees y_k = x_k + v_k; the plant runs on plant_params (16x1 | 16xS, [] = params) under
         * plant_profile, plus the disturbance w_k.  w, v: 2 x k_sim x S (or 2k_sim x S), [] = none.  xk holds the
         * true states. */
        int S, N, k_sim, i_sim, profile, pprofile, pc, ppc, i;
        double eps;
        const double *pp = NULL, *w = NULL, *v = NULL;
        mxArray *xk, *uk, *cost, *inner, *status;
        int *ibuf;
        if (nrhs != 11)
            mexErrMsgIdAndTxt("ntm:arg", "usage: [xk,uk,cost,inner,status] = ntm_mpc_batch_perturbed(x0, params, N, k_sim, i_sim, eps, profile, plant_params, plant_profile, w, v)");
        S = states_arg(prhs[0]);
        if (!is_real_double(prhs[1]) || mxGetM(prhs[1]) != NTM_NPARAM || ((int)mxGetN(prhs[1]) != 1 && (int)mxGetN(prhs[1]) != S))
            mexErrMsgIdAndTxt("ntm:arg", "params must be 16 x 1 or 16 x S (see ntm_mpc.h)");
        pc = (int)mxGetN(prhs[1]);
        N = (int)scalar_arg(nrhs, prhs, 2, ""); k_sim = (int)scalar_arg(nrhs, prhs, 3, ""); i_sim = (int)scalar_arg(nrhs, prhs, 4, "");
        eps = scalar_arg(nrhs, prhs, 5, ""); profile = (int)scalar_arg(nrhs, prhs, 6, "");
        pprofile = (int)scalar_arg(nrhs, prhs, 8, "");
        if (N < 1 || N > NTM_MAX_HORIZON || k_sim < 0 || i_sim < 1) mexErrMsgIdAndTxt("ntm:arg", "N in 1..128, k_sim >= 0, i_sim >= 1");
        if (profile & NTM_PROFILE_TAUE_W) mexErrMsgIdAndTxt("ntm:arg", "NTM_PROFILE_TAUE_W (128) is not supported on the controller side");
        if (pprofile & ~(NTM_PROFILE_RHO1_SQ | NTM_PROFILE_PLANT_C | NTM_PROFILE_PLANT_RK4 | NTM_PROFILE_TAUE_W))
            mexErrMsgIdAndTxt("ntm:arg", "plant_profile: only RHO1_SQ, PLANT_C, PLANT_RK4 and TAUE_W (1, 8, 64, 128) act on the plant");
        ppc = pc;
        if (mxGetNumberOfElements(prhs[7]) != 0) {
            if (!is_real_double(prhs[7]) || mxGetM(prhs[7]) != NTM_NPARAM || ((int)mxGetN(prhs[7]) != 1 && (int)mxGetN(prhs[7]) != S))
                mexErrMsgIdAndTxt("ntm:arg", "plant_params must be [], 16 x 1 or 16 x S");
            pp = mxGetPr(prhs[7]); ppc = (int)mxGetN(prhs[7]);
        }
        for (i = 9; i <= 10; ++i) {
            if (mxGetNumberOfElements(prhs[i]) == 0) continue;
            if (!is_real_double(prhs[i]) || mxGetNumberOfElements(prhs[i]) != 2 * (size_t)k_sim * S)
                mexErrMsgIdAndTxt("ntm:arg", "w and v must be [] or real doubles of 2 x k_sim x S");
            if (i == 9) w = mxGetPr(prhs[i]); else v = mxGetPr(prhs[i]);
        }
        xk = mxCreateDoubleMatrix(2 * (k_sim + 1), S, mxREAL); uk = mxCreateDoubleMatrix(k_sim, S, mxREAL);
        cost = mxCreateDoubleMatrix(1, S, mxREAL); inner = mxCreateDoubleMatrix(k_sim, S, mxREAL); status = mxCreateDoubleMatrix(1, S, mxREAL);
        ibuf = (int *)mxMalloc(sizeof(int) * ((size_t)k_sim * S + S + 1));
        check(ntm_mpc_closed_loop_perturbed(handle(), NTM_LAYOUT_MATLAB, profile, S, N, k_sim, i_sim, eps, mxGetPr(prhs[0]),
                                            mxGetPr(prhs[1]), pc, pp, ppc, pprofile, w, v, mxGetPr(xk), mxGetPr(uk), NULL,
                                            mxGetPr(cost), ibuf, NULL, ibuf + (size_t)k_sim * S));
        for (i = 0; i < k_sim * S; ++i) mxGetPr(inner)[i] = (double)ibuf[i];
        for (i = 0; i < S; ++i) mxGetPr(status)[i] = (double)ibuf[(size_t)k_sim * S + i];
        mxFree(ibuf);
        plhs[0] = xk;
        if (nlhs > 1) plhs[1] = uk; else mxDestroyArray(uk);
        if (nlhs > 2) plhs[2] = cost; else mxDestroyArray(cost);
        if (nlhs > 3) plhs[3] = inner; else mxDestroyArray(inner);
        if (nlhs > 4) plhs[4] = status; else mxDestroyArray(status);
    }
#else
#error "unknown NTM_MEX_FN"
#endif
}
