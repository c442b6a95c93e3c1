"""NumPy twin of ``ntm_mpc_closed_loop_perturbed_sc`` (TEST INFRASTRUCTURE ONLY): the state-row controller step of
``tests/controller_sc_oracle.py`` at the measured state, the oracle's ``plant_step`` on the plant's own physics and
profile, plus the disturbance.  Both primitives are used unchanged, so the twin IS the step-API composition.  A step that
comes back infeasible ends the scenario as ``oracle.closed_loop(state_rows=...)`` does."""
from __future__ import annotations

import numpy as np

from controller_sc_oracle import controller_step_sc
from oracle import ntm_oracle as o


def closed_loop_perturbed_sc(p, x0, N: int = 3, k_sim: int = 20, i_sim: int = 10, eps: float = 1e-14,
                             profile: o.Profile = o.LITERAL, state_rows: int = o.STATE_ROWS_REFRESH, xbounds=None,
                             plant_p=None, plant_profile: o.Profile = None, d=None, v=None):
    """One scenario: ``y_k = x_k + v[k]``, ``u_k = controller_step_sc(p, ..., y_k)``, ``x_{k+1} = plant_step(plant_p,
    x_k, u_k, plant_profile) + d[k]``.  ``d`` / ``v``: ``[k_sim, 2]`` or None, ``plant_p`` defaults to ``p`` and
    ``plant_profile`` to ``profile``.  Returns the dict of ``o.closed_loop`` plus ``k_inf`` (the infeasible step, or
    None): up to and including that step, the composition's outputs (NaN u and U and the step's iteration counts at
    it); after it, uk, Uk and xk(:, k_inf+1 ..) NaN, iteration counts 0, cost NaN, status 3."""
    plant_p = p if plant_p is None else plant_p
    plant_profile = profile if plant_profile is None else plant_profile
    state, x = {}, np.asarray(x0, dtype=np.float64).ravel().copy()
    xk = np.full((2, k_sim + 1), np.nan); xk[:, 0] = x
    uk = np.full(k_sim, np.nan); Uk = np.full((N, k_sim), np.nan)
    inner = np.zeros(k_sim, dtype=np.int32); qpit = np.zeros(k_sim, dtype=np.int32)
    status, k_inf = 0, None
    with np.errstate(all="ignore"):
        for k in range(k_sim):
            y = x if v is None else x + v[k]
            r = controller_step_sc(p, state, y, N, i_sim, eps, profile, state_rows=state_rows, xbounds=xbounds)
            inner[k], qpit[k] = r["inner_iters"], r["qp_iters"]
            status = max(status, r["status"])
            if r["status"] == o.QP_INFEASIBLE:
                k_inf = k
                break
            x = o.plant_step(plant_p, x, r["u"], plant_profile)
            if d is not None:
                x = x + d[k]
            xk[:, k + 1] = x; uk[k] = r["u"]; Uk[:, k] = r["U"]
    if not np.all(np.isfinite(xk)):
        status = max(status, 2)
    if k_inf is not None:
        return dict(xk=xk, uk=uk, Uk=Uk, inner_iters=inner, qp_iters=qpit, cost=float("nan"), status=status, k_inf=k_inf)
    rr = np.array([p["r1"], p["r2"]]); Q = np.array([[p["q11"], p["q12"]], [p["q12"], p["q22"]]])
    e = xk[:, 1:] - rr[:, None]
    return dict(xk=xk, uk=uk, Uk=Uk, inner_iters=inner, qp_iters=qpit, cost=float(np.sum(e * (Q @ e))), status=status,
                k_inf=None)
