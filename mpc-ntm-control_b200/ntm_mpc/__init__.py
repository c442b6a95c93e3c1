"""ntm_mpc -- host side of the B200-native LPV-MPC hot path of IsaacSavona/MPC-NTM-Control.

Everything numerical runs in lib/libntm_mpc.so (hand-written sm_100a CUDA behind the C ABI of
include/ntm_mpc.h).  Importing this package does not need a GPU; calling it does.
"""
from . import montecarlo, physics, plots  # noqa: F401
from ._lib import (LAYOUT_MATLAB, LAYOUT_SOA, MAX_HORIZON, NPARAM, PROFILE_CONSISTENT, PROFILE_DENSE_G,  # noqa: F401
                   PROFILE_F_XK, PROFILE_GAMMA_I, PROFILE_INNER_FIXED, PROFILE_LITERAL, PROFILE_PLANT_C,
                   PROFILE_PLANT_RK4, PROFILE_RHO1_SQ, PROFILE_TAUE_W, STATE_ROWS_FROZEN, STATE_ROWS_OFF, STATE_ROWS_REFRESH, NtmError)
from ._lib import ctrl_doubles, rec_doubles  # noqa: F401
from .api import Controller, NtmMpc, closed_loop_multi, device_count  # noqa: F401
from .reference_api import (A, B, LpvA, LpvB, NTM_MPC_Sim, Rho_to_PhiGammaLambda, bind_workspace, getWLc,  # noqa: F401
                            quadprog, rho1, rho2, rho3, workspace_from_physics)
