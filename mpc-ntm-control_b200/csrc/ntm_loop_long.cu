// ntm_loop_long.cu -- long-horizon (33 <= N <= 128) instantiations of the fused closed loop, literal Gamma, EC-power box
// QP: closed_loop_kernel<GW, false, 0|1|3> on the packed sweep tableau (ntm_long.cuh).  One CTA of GW warps per scenario,
// ~60 KB of shared memory at N = 100, three CTAs per SM (round 1: 178 KB, one CTA per SM).
#include "ntm_loop.cuh"

namespace ntm {

template <int GW, int EXT, int LV, bool CTL = false>
static cudaError_t launch_long(cudaStream_t st, const DeviceProps &dp, const LoopArgs &a) {
    const size_t smem = work_bytes_long(a.N);
    if (smem > dp.smem_optin) return cudaErrorInvalidConfiguration;
    static thread_local size_t c_smem = 0;
    static thread_local int c_occ = 0, c_dev = -1;
    int dev = 0;
    cudaGetDevice(&dev);
    if (c_smem != smem || c_dev != dev) {
        cudaError_t e = raise_smem_attribute(reinterpret_cast<const void *>(closed_loop_kernel<GW, false, EXT, LV, CTL>), dev, dp.smem_optin);
        if (e != cudaSuccess) return e;
        int occ = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, closed_loop_kernel<GW, false, EXT, LV, CTL>, 32 * GW, smem);
        if (e != cudaSuccess) return e;
        c_smem = smem; c_occ = occ; c_dev = dev;
    }
    if (c_occ < 1) return cudaErrorInvalidConfiguration;
    long long grid = (long long)c_occ * dp.sm_count;
    if (grid > a.S) grid = a.S;
    closed_loop_kernel<GW, false, EXT, LV, CTL><<<(int)grid, 32 * GW, smem, st>>>(a, (unsigned int)smem);
    return cudaGetLastError();
}

cudaError_t launch_closed_loop_long(cudaStream_t st, const DeviceProps &dp, const LoopArgs &a, long long *launches) {
    const bool rk4 = (a.flags & (NTM_PROFILE_PLANT_RK4 | NTM_PROFILE_TAUE_W)) != 0;   // the EXT = 1 instantiations: cold plant options
    cudaError_t e;
    // tableau in registers: 7 x 7 blocks, thread I(I+1)/2 + J owns block (I, J): N + 1 <= 70 (2 warps) / 105 (4 warps)
    if (a.pert) {                                          // perturbed plant (EXT = 3): its own instantiations
        if (a.N <= 64) e = launch_long<2, 3, 0>(st, dp, a);
        else if (a.N + 1 <= NTM_TS * 15) e = launch_long<4, 3, 0>(st, dp, a);
        else e = launch_long<4, 3, 1>(st, dp, a);
    } else if (a.ctl) {                                           // controller step (EXT = 0): its own instantiations
        if (a.N <= 64) e = launch_long<2, 0, 0, true>(st, dp, a);
        else if (a.N + 1 <= NTM_TS * 15) e = launch_long<4, 0, 0, true>(st, dp, a);
        else e = launch_long<4, 0, 1, true>(st, dp, a);
    } else if (a.N <= 64) e = rk4 ? launch_long<2, 1, 0>(st, dp, a) : launch_long<2, 0, 0>(st, dp, a);
    else if (a.N + 1 <= NTM_TS * 15) e = rk4 ? launch_long<4, 1, 0>(st, dp, a) : launch_long<4, 0, 0>(st, dp, a);
    else e = rk4 ? launch_long<4, 1, 1>(st, dp, a) : launch_long<4, 0, 1>(st, dp, a);
    if (e == cudaSuccess) ++*launches;
    return e;
}

}  // namespace ntm
