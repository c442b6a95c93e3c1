// ntm_kernels.h -- host-side launch interface between the C ABI (ntm_cabi.cu) and the kernels.
#pragma once
#include <cstddef>
#include <cuda_runtime.h>

namespace ntm {

// The perturbed plant's inputs (ntm_mpc_closed_loop_perturbed[_sc]): the plant runs on its own parameter block
// (pparams_count 1 or S, `layout`) and profile bits pflags; the controller sees x_k + v_k, the plant adds d_k after its
// step.  dist (d) / noise (v): 2 * k_sim doubles per scenario in `layout`, element 2k + i (NULL = none)
struct PlantIn {
    const double *pparams, *dist, *noise;
    int pparams_count, pflags;
};

// The LPV Kalman filter's covariances (ntm_kf_step, kf_cov of include/ntm_mpc.h): Qw and Rv, lower triangles
struct KfCov {
    double q11, q21, q22, r11, r21, r22;
};

// The observer of ntm_mpc_closed_loop_observed: the controller sees the estimate of one ntm_kf_step per time step.
// rec: NTM_KF_DOUBLES per scenario, scenario slowest (handle-owned scratch); xhat: 2 * k_sim doubles
// per scenario in `layout`, element 2k + i (or NULL); mflags: the model bits of the controller's profile word
// (RHO1_SQ | PLANT_C | PLANT_RK4), taken before check_fused strips the plant bits from `flags`; on (host only): the
// call has an observer, and the C ABI layer points rec at the handle's scratch.
struct ObsIn {
    double *rec, *xhat;
    KfCov cov;
    int mflags, on;
};

struct LoopArgs {
    int layout, flags, S, N, k_sim, i_sim;
    double eps;
    const double *x0, *params;
    int params_count;
    double *xk, *uk, *Uk, *cost;
    int *inner, *qpit, *status;
    unsigned int *counter;   // work-queue head, zeroed before the launch
    int hcap;                // shared-memory LDL' capacity (set by the launcher)
    int gam;                 // 1: the work area carries a dense-Gamma staging tile (set by the launcher)
    double *hscratch;        // global LDL' slabs, one per resident group, for free sets larger than the smem workspace
    // state rows of getWLc.m inside the loop (SURVEY 8f-1): 0 = dropped (box QP), 1 = rebuilt from every
    // re-condensation, 2 = frozen at the offline build as NTM_MPC_Sim.m:74 literally does
    int srows;
    double xmin1, xmax1, xmin2, xmax2;   // the state box of the state rows, NTM_MPC_Sim.m:44-45
    PlantIn pp;                          // the perturbed plant's inputs (pert = 1)
    unsigned int wbytes, qbytes;         // offsets of the IneqWork / ExtWork areas in a group's shared memory (launcher)
    int rows_warm;                       // 1: state-row QPs on the literal Gamma start from an earlier active set (the dense
                                         // Gamma always starts cold); set by the launcher, NTM_ROWS_WARM=0 turns it off
    // packed-record output (the multi-GPU gather wants ONE contiguous block per scenario): when rec_ld > 0, xk / uk /
    // cost / rec_status point INTO one array of rec_ld doubles per scenario (scenario slowest) instead of three arrays
    int rec_ld;
    double *rec_status;                  // record mode: the status word as a double (0..3), or NULL
    // Two-phase launch with a longest-first work queue (one-warp box loop, see lpt_doubles): phase A runs time step 0 of
    // every scenario, saves its loop state (one controller record per scenario in sv) and a cost key (how many of the
    // step's QPs missed the vertex test); a counting sort turns the keys into the order in which phase B pops the
    // scenarios for the remaining steps.  A launch is as long as its slowest scenario STARTED LAST, and the slow scenarios
    // are slow in every step.  sv (and launch_closed_loop's lpt): buffers from the C ABI layer (NULL = one launch in
    // natural order); the rest is set by the launcher.
    double *sv;                          // NTM_CTRL_DOUBLES(N) per scenario (include/ntm_mpc.h), scenario slowest
    int k_begin, k_end;                  // time steps [k_begin, k_end) of this launch
    int *lpt_key;                        // phase A
    const int *perm;                     // phase B
    // controller step (ntm_mpc_step[_sc]): k_sim = 1, x0 is the measured state, sv holds the caller's records (read at
    // the start, written at the stop rule), no plant; xk and cost are NULL
    int ctl;
    int pert;                            // 1: perturbed plant (ntm_mpc_closed_loop_perturbed[_sc], see `pp` above)
    ObsIn obs;                           // the observer of ntm_mpc_closed_loop_observed (pert = 1, obs.on = 1)
};
#define NTM_LPT_BINS 160

struct DeviceProps {
    int sm_count, cc_major, cc_minor;
    size_t smem_optin;
};

// bytes of global LDL' scratch (one N x (N|1) slab per group that can be resident) for horizon N on this device
size_t hscratch_bytes(const DeviceProps &dp, int N);
// two-phase launch: doubles of LoopArgs::sv this launch would use (0: one launch in natural order); lpt needs
// 2 S + NTM_LPT_BINS ints
size_t lpt_doubles(const DeviceProps &dp, const LoopArgs &a);
// dynamic shared memory per CTA of the fused kernel with the state rows of getWLc.m kept (LoopArgs::srows != 0)
size_t state_rows_smem(int N);
// the same for ONE group with a non-literal Gamma index (NTM_PROFILE_GAMMA_I / DENSE_G; one-warp groups, N <= 32)
size_t state_rows_dense_smem(int N, int srows);
// groups per CTA of the general-inequality QP (launch_qp_ineq) whose N x N factor pair + row scales fit in shared memory;
// 0: not even one fits
int qp_ineq_groups(const DeviceProps &dp, int N, int M);

// every launcher returns the CUDA error of the launch (cudaSuccess on success) and adds the number of
// kernels it launched to *launches
cudaError_t launch_rho(cudaStream_t st, int layout, int flags, int S, const double *x, const double *params,
                       int pc, double *r1, double *r2, double *r3, long long *launches);
cudaError_t launch_lpv(cudaStream_t st, int layout, int S, const double *r1, const double *r2, const double *r3,
                       const double *params, int pc, double *A, double *B, long long *launches);
cudaError_t launch_plant(cudaStream_t st, int layout, int flags, int S, const double *x, const double *u,
                         const double *params, int pc, double *xn, long long *launches);
// one ntm_kf_step: rec (NTM_KF_DOUBLES per scenario, scenario slowest) in place, xhat[2 * S] in `layout` (or NULL)
cudaError_t launch_kf(cudaStream_t st, int layout, int mflags, int S, const double *y, const double *u,
                      const double *params, int pc, const KfCov &cov, double *rec, double *xhat, long long *launches);
cudaError_t launch_condense(cudaStream_t st, const DeviceProps &dp, int layout, int flags, int S, int N,
                            const double *R1, const double *R2, const double *R3, const double *params, int pc,
                            double *Phi, double *Gam, double *Lam, long long *launches);
cudaError_t launch_hessian_grad(cudaStream_t st, const DeviceProps &dp, int layout, int S, int N, const double *Phi,
                                const double *Gam, const double *Lam, const double *x, const double *params, int pc,
                                double *G, double *F, long long *launches);
cudaError_t launch_qp_box(cudaStream_t st, const DeviceProps &dp, int layout, int S, int N, const double *G,
                          const double *F, const double *lb, const double *ub, int bc, double *U, int *iters,
                          int *status, unsigned int *counter, double *hscratch, long long *launches);
cudaError_t launch_qp_ineq(cudaStream_t st, const DeviceProps &dp, int layout, int S, int N, int M, const double *G,
                           const double *F, const double *lb, const double *ub, int bc, const double *Lg,
                           const double *bg, double *U, int *iters, int *status, unsigned int *counter,
                           long long *launches);
cudaError_t launch_getwlc(cudaStream_t st, const DeviceProps &dp, int layout, int S, int N, const double *bounds,
                          const double *Gam, const double *Phi, const double *Lam, double *W, double *L, double *c,
                          long long *launches);
// umin / umax of scenario s: umin[s * ustride], umax[s * ustride] (ustride 0 = one shared pair)
cudaError_t launch_mc_stats(cudaStream_t st, const DeviceProps &dp, int layout, int S, int k_sim, const double *xk,
                            const double *uk, const double *cost, const int *status, const double *umin, const double *umax,
                            int ustride, const double *bounds, double w_sup, double hist_max, double *out, long long *launches);
// lpt: the two-phase launch's keys, order and bins (2 S + NTM_LPT_BINS ints; used when a.sv is set and lpt_doubles is
// not 0), or NULL
cudaError_t launch_closed_loop(cudaStream_t st, const DeviceProps &dp, const LoopArgs &a, int *lpt, long long *launches);

// EXT template argument of closed_loop_kernel: the instantiation key; what each one carries is spelled out by the
// members of LoopTraits (ntm_loop.cuh)
constexpr int EXT_BOX = 0;
constexpr int EXT_COLD_PLANT = 1;
constexpr int EXT_STATE_ROWS = 2;
constexpr int EXT_PERTURBED = 3;
constexpr int EXT_PERTURBED_ROWS = 4;
constexpr int EXT_OBSERVED = 5;          // EXT_PERTURBED + the observer (LoopArgs::obs)
constexpr int EXT_OBSERVED_ROWS = 6;     // EXT_PERTURBED_ROWS + the observer
// one instantiation closed_loop_kernel<gw, dense, ext, lv, ctl>
struct LoopKey {
    int gw;
    bool dense;
    int ext, lv;
    bool ctl;
};
using LoopKernelFn = void (*)(LoopArgs, unsigned int);
struct LoopKernel {
    LoopKey key;
    LoopKernelFn fn;
};
template <int N>
inline LoopKernelFn find_loop_kernel(const LoopKernel (&table)[N], const LoopKey &k) {
    for (const LoopKernel &t : table)
        if (t.key.gw == k.gw && t.key.dense == k.dense && t.key.ext == k.ext && t.key.lv == k.lv && t.key.ctl == k.ctl) return t.fn;
    return nullptr;
}
// the long-horizon instantiations (N > 32, literal Gamma, box QP), compiled in ntm_loop_long.cu
LoopKernelFn find_long_loop_kernel(const LoopKey &k);
// raises cudaFuncAttributeMaxDynamicSharedMemorySize of a kernel to the device maximum, once per (kernel, device)
cudaError_t raise_smem_attribute(const void *fn, int dev, size_t smem_optin);
cudaError_t launch_fp64_peak(cudaStream_t st, const DeviceProps &dp, int iters, double *out, long long *launches);
cudaError_t launch_dmma_peak(cudaStream_t st, const DeviceProps &dp, int iters, double *out, long long *launches);

}  // namespace ntm
