"""NumPy restatement of ONE controller step with getWLc's state rows kept, the twin of ``ntm_mpc_step_sc`` (TEST
INFRASTRUCTURE ONLY).

Built on ``controller_step`` of ``tests/controller_oracle.py`` (the box-QP step, unchanged) with ``o.qp_state_rows`` as its
QP, so both twins share one restatement of NTM_MPC_Sim.m:94-128.  ``tests/test_controller_sc_cpu.py`` keeps this twin and
``oracle.closed_loop(state_rows=...)`` from drifting apart."""
from __future__ import annotations

import copy

import numpy as np

from controller_oracle import controller_step
from oracle import ntm_oracle as o


class _Infeasible(Exception):
    """quadprog exitflag -2 (:100-101): the step ends without a U."""


def controller_step_sc(p, state: dict, x, N: int = 3, i_sim: int = 10, eps: float = 1e-14,
                       profile: o.Profile = o.LITERAL, state_rows: int = o.STATE_ROWS_REFRESH, xbounds=None):
    """``controller_step`` with the QP of :97 as written: ``quadprog(G, F, L, c + W*xk(:,k))`` with getWLc's state rows.

    ``state_rows`` / ``xbounds = (xmin1, xmax1, xmin2, xmax2)`` as in ``oracle.closed_loop``.  REFRESH rows come from the
    condensation of the stage entries on hand (the last re-condensation, :119); FROZEN rows from the offline build, kept
    in ``state["rows"]`` (:74).  Stepped with ``plant_step``, it reproduces ``closed_loop(state_rows=...)`` up to the
    step at which a scenario turns infeasible.  An infeasible QP returns NaN u and U, status 3, the iteration counts of
    that step, and leaves ``state`` exactly as it was before the call."""
    if state_rows == o.STATE_ROWS_OFF:
        return controller_step(p, state, x, N, i_sim, eps, profile)
    Af, Bf, C = o.model_callables(p)
    xv = np.asarray(x, dtype=np.float64).ravel()
    xmin = np.array([xbounds[0], xbounds[2]]); xmax = np.array([xbounds[1], xbounds[3]])
    before = copy.deepcopy(state)
    seen = dict(calls=0, nit=0, status=0)

    def condensed():
        # controller_step re-schedules state["Rho1..3"] in place (:114-117): at every QP they hold the stage entries
        # the G, F on hand were built from
        return o.Rho_to_PhiGammaLambda(state["Rho1"], state["Rho2"], state["Rho3"], Af, Bf, C, profile.gamma_index)

    def qp(G, F, lb, ub):
        if state_rows == o.STATE_ROWS_FROZEN:
            if "rows" not in state:                    # first QP of a fresh controller: the offline stage entries
                state["rows"] = condensed()
            rows = state["rows"]
        else:
            rows = condensed()
        U, nit, st = o.qp_state_rows(G, F, lb, ub, *rows, xv, xmin, xmax)
        seen["calls"] += 1; seen["nit"] += nit; seen["status"] = max(seen["status"], st)
        if st == o.QP_INFEASIBLE:
            raise _Infeasible
        return U, nit, st

    try:
        return controller_step(p, state, x, N, i_sim, eps, profile, qp=qp)
    except _Infeasible:
        state.clear()
        state.update(before)
        return dict(u=float("nan"), U=np.full(N, np.nan), inner_iters=seen["calls"], qp_iters=seen["nit"],
                    status=seen["status"])
