"""NumPy twin of the state observer (TEST INFRASTRUCTURE ONLY): one step of ``ntm_kf_step`` and
``ntm_mpc_closed_loop_observed`` composed from it, the controller twins of ``tests/controller_sc_oracle.py`` (the box-QP
step of ``tests/controller_oracle.py`` with the rows off) and the oracle's ``plant_step``.  The filter is written with
matrix products; the device restates it with explicit roundings, so the two agree to rounding, not bit for bit."""
from __future__ import annotations

import numpy as np

from controller_sc_oracle import controller_step_sc
from oracle import ntm_oracle as o

KF_DOUBLES = 6


def model_profile(profile: o.Profile) -> o.Profile:
    """The plant the filter predicts with: the RHO1_SQ, PLANT_C and PLANT_RK4 choices of the controller's profile."""
    return o.Profile(rho1_variant=profile.rho1_variant, plant_affine=profile.plant_affine,
                     plant_integrator=profile.plant_integrator)


def covariances(kf_cov):
    """``(Qw, Rv)`` as symmetric 2 x 2 matrices from ``kf_cov = (qw11, qw21, qw22, rv11, rv21, rv22)``."""
    q11, q21, q22, r11, r21, r22 = np.asarray(kf_cov, dtype=np.float64).ravel()
    return np.array([[q11, q21], [q21, q22]]), np.array([[r11, r21], [r21, r22]])


def kf_step(p, rec, y, u, kf_cov, profile: o.Profile = o.LITERAL) -> np.ndarray:
    """One step of the quasi-LPV Kalman filter on one record ``rec`` (xhat, p11, p21, p22, steps); returns the new
    record.  Fresh (steps == 0): xhat = y, P = Rv.  Otherwise xhat- = plant_step(xhat, u), F = A(rho(xhat)) of A.m:2,
    P- = F P F' + Qw, K = P- (P- + Rv)^-1, xhat = xhat- + K (y - xhat-), P = (I - K) P- (I - K)' + K Rv K'."""
    Qw, Rv = covariances(kf_cov)
    rec = np.asarray(rec, dtype=np.float64).ravel()
    y = np.asarray(y, dtype=np.float64).ravel()
    if rec[5] == 0.0:
        return np.array([y[0], y[1], Rv[0, 0], Rv[1, 0], Rv[1, 1], 1.0])
    xh = rec[:2]
    P = np.array([[rec[2], rec[3]], [rec[3], rec[4]]])
    with np.errstate(all="ignore"):
        xm = o.plant_step(p, xh, u, model_profile(profile))
        Af, _, _ = o.model_callables(p)
        F = Af(o.rho1(xh, p["w_marg"], profile.rho1_variant), o.rho2(xh))
        Pm = F @ P @ F.T + Qw
        Sg = Pm + Rv
        det = Sg[0, 0] * Sg[1, 1] - Sg[1, 0] * Sg[0, 1]
        K = Pm @ (np.array([[Sg[1, 1], -Sg[0, 1]], [-Sg[1, 0], Sg[0, 0]]]) / det)
        xn = xm + K @ (y - xm)
        IK = np.eye(2) - K
        Pn = IK @ Pm @ IK.T + K @ Rv @ K.T
    return np.array([xn[0], xn[1], Pn[0, 0], 0.5 * (Pn[1, 0] + Pn[0, 1]), Pn[1, 1], rec[5] + 1.0])


def closed_loop_observed(p, x0, N: int = 3, k_sim: int = 20, i_sim: int = 10, eps: float = 1e-14,
                         profile: o.Profile = o.LITERAL, state_rows: int = o.STATE_ROWS_OFF, xbounds=None, plant_p=None,
                         plant_profile: o.Profile = None, d=None, v=None, kf_cov=None):
    """One scenario: ``y_k = x_k + v[k]``, ``xhat_k = kf_step(y_k, u_{k-1})`` (fresh at k = 0),
    ``u_k = controller_step_sc(p, ..., xhat_k)``, ``x_{k+1} = plant_step(plant_p, x_k, u_k, plant_profile) + d[k]``.
    Returns the dict of ``perturbed_sc_oracle.closed_loop_perturbed_sc`` plus ``xhat`` (2, k_sim) and the final filter
    record ``kf``; after an infeasible step xhat is NaN."""
    plant_p = p if plant_p is None else plant_p
    plant_profile = profile if plant_profile is None else plant_profile
    state, x = {}, np.asarray(x0, dtype=np.float64).ravel().copy()
    kf = np.zeros(KF_DOUBLES)
    xk = np.full((2, k_sim + 1), np.nan); xk[:, 0] = x
    xhat = np.full((2, k_sim), np.nan)
    uk = np.full(k_sim, np.nan); Uk = np.full((N, k_sim), np.nan)
    inner = np.zeros(k_sim, dtype=np.int32); qpit = np.zeros(k_sim, dtype=np.int32)
    status, k_inf, u_prev = 0, None, 0.0
    with np.errstate(all="ignore"):
        for k in range(k_sim):
            y = x if v is None else x + v[k]
            kf = kf_step(p, kf, y, u_prev, kf_cov, profile)
            xhat[:, k] = kf[:2]
            r = controller_step_sc(p, state, kf[:2].copy(), N, i_sim, eps, profile, state_rows=state_rows,
                                   xbounds=xbounds)
            inner[k], qpit[k] = r["inner_iters"], r["qp_iters"]
            status = max(status, r["status"])
            if r["status"] == o.QP_INFEASIBLE:
                k_inf = k
                break
            x = o.plant_step(plant_p, x, r["u"], plant_profile)
            if d is not None:
                x = x + d[k]
            xk[:, k + 1] = x; uk[k] = r["u"]; Uk[:, k] = r["U"]; u_prev = r["u"]
    if not np.all(np.isfinite(xk)):
        status = max(status, 2)
    res = dict(xk=xk, uk=uk, Uk=Uk, inner_iters=inner, qp_iters=qpit, status=status, k_inf=k_inf, xhat=xhat, kf=kf)
    if k_inf is not None:
        res["cost"] = float("nan")
        return res
    rr = np.array([p["r1"], p["r2"]]); Q = np.array([[p["q11"], p["q12"]], [p["q12"], p["q22"]]])
    e = xk[:, 1:] - rr[:, None]
    res["cost"] = float(np.sum(e * (Q @ e)))
    return res
