"""NumPy twin of ``ntm_mpc_closed_loop_perturbed`` (TEST INFRASTRUCTURE ONLY): the controller step of
``tests/controller_oracle.py`` at the measured state, the oracle's ``plant_step`` on the plant's own physics and
profile, plus the disturbance.  Both primitives are used unchanged, so the twin IS the step-API composition."""
from __future__ import annotations

import numpy as np

from controller_oracle import controller_step
from oracle import ntm_oracle as o


def closed_loop_perturbed(p, x0, N: int = 3, k_sim: int = 20, i_sim: int = 10, eps: float = 1e-14,
                          profile: o.Profile = o.LITERAL, plant_p=None, plant_profile: o.Profile = None, d=None, v=None):
    """One scenario: ``y_k = x_k + v[k]``, ``u_k = controller_step(p, ..., y_k)``, ``x_{k+1} = plant_step(plant_p, x_k,
    u_k, plant_profile) + d[k]``.  ``d`` / ``v``: ``[k_sim, 2]`` or None (no add), ``plant_p`` defaults to ``p`` and
    ``plant_profile`` to ``profile``.  Returns the dict of ``o.closed_loop``: ``xk`` holds the true states, ``cost`` is
    judged on them with the controller's r and Q, ``status`` is the worst over the run (2 for a non-finite y, u or x)."""
    plant_p = p if plant_p is None else plant_p
    plant_profile = profile if plant_profile is None else plant_profile
    state, x = {}, np.asarray(x0, dtype=np.float64).ravel().copy()
    xk, uk, Uk, inner, qpit, status = [x], [], [], [], [], 0
    with np.errstate(all="ignore"):
        for k in range(k_sim):
            y = x if v is None else x + v[k]
            r = controller_step(p, state, y, N, i_sim, eps, profile)
            x = o.plant_step(plant_p, x, r["u"], plant_profile)
            if d is not None:
                x = x + d[k]
            xk.append(x); uk.append(r["u"]); Uk.append(r["U"])
            inner.append(r["inner_iters"]); qpit.append(r["qp_iters"]); status = max(status, r["status"])
    xk = np.array(xk).T
    if not np.all(np.isfinite(xk)):
        status = max(status, 2)
    rr = np.array([p["r1"], p["r2"]]); Q = np.array([[p["q11"], p["q12"]], [p["q12"], p["q22"]]])
    e = xk[:, 1:] - rr[:, None]
    return dict(xk=xk, uk=np.array(uk), Uk=np.array(Uk).T.reshape(N, k_sim), inner_iters=np.array(inner, dtype=np.int32),
                qp_iters=np.array(qpit, dtype=np.int32), cost=float(np.sum(e * (Q @ e))), status=status)
