// ntm_loop_long.cu -- long-horizon (33 <= N <= 128) instantiations of the fused closed loop, literal Gamma, EC-power box
// QP: closed_loop_kernel<GW, false, EXT_BOX | EXT_COLD_PLANT | EXT_PERTURBED> on the packed sweep tableau (ntm_long.cuh).
// One CTA of GW warps per scenario, ~60 KB of shared memory at N = 100, three CTAs per SM (round 1: 178 KB, one CTA per
// SM).  Which one runs, and its launch shape: route_closed_loop (ntm_kernels.cu).
#include "ntm_loop.cuh"

namespace ntm {

// LV = 0: the tableau in registers, 7 x 7 blocks, thread I(I+1)/2 + J owns block (I, J): N + 1 <= 70 (2 warps) / 105 (4)
static const LoopKernel kLongLoopKernels[] = {
    {{2, false, EXT_BOX, 0, false}, closed_loop_kernel<2, false, EXT_BOX, 0>},
    {{4, false, EXT_BOX, 0, false}, closed_loop_kernel<4, false, EXT_BOX, 0>},
    {{4, false, EXT_BOX, 1, false}, closed_loop_kernel<4, false, EXT_BOX, 1>},
    {{2, false, EXT_COLD_PLANT, 0, false}, closed_loop_kernel<2, false, EXT_COLD_PLANT, 0>},
    {{4, false, EXT_COLD_PLANT, 0, false}, closed_loop_kernel<4, false, EXT_COLD_PLANT, 0>},
    {{4, false, EXT_COLD_PLANT, 1, false}, closed_loop_kernel<4, false, EXT_COLD_PLANT, 1>},
    {{2, false, EXT_PERTURBED, 0, false}, closed_loop_kernel<2, false, EXT_PERTURBED, 0>},
    {{4, false, EXT_PERTURBED, 0, false}, closed_loop_kernel<4, false, EXT_PERTURBED, 0>},
    {{4, false, EXT_PERTURBED, 1, false}, closed_loop_kernel<4, false, EXT_PERTURBED, 1>},
    {{2, false, EXT_BOX, 0, true}, closed_loop_kernel<2, false, EXT_BOX, 0, true>},   // controller step
    {{4, false, EXT_BOX, 0, true}, closed_loop_kernel<4, false, EXT_BOX, 0, true>},
    {{4, false, EXT_BOX, 1, true}, closed_loop_kernel<4, false, EXT_BOX, 1, true>},
};

LoopKernelFn find_long_loop_kernel(const LoopKey &k) { return find_loop_kernel(kLongLoopKernels, k); }

}  // namespace ntm
