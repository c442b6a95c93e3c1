"""NumPy restatement of ONE controller step, the twin of ``ntm_mpc_step`` (TEST INFRASTRUCTURE ONLY).

Built from the primitives of ``oracle/ntm_oracle.py`` and kept beside the tests that use it: the oracle module, its golden
fixtures and the 50-digit adjudication tools stay pinned to ``closed_loop`` exactly as it is.
``tests/test_controller_cpu.py`` keeps this restatement and ``closed_loop`` from drifting apart."""
from __future__ import annotations

from typing import Callable

import numpy as np

from oracle import ntm_oracle as o


def controller_step(p, state: dict, x, N: int = 3, i_sim: int = 10, eps: float = 1e-14, profile: o.Profile = o.LITERAL,
                    qp: Callable = o.qp_box):
    """One pass of NTM_MPC_Sim.m:94-128 (no plant) at the measured state ``x``: the restatement of ``ntm_mpc_step``.

    ``state`` is a dict updated in place; an empty dict is a fresh controller, whose first step runs the offline build
    :63-73 from ``x`` (which becomes ``x0``).  It carries what crosses a time step of ``closed_loop``: Rho1..3, Uold,
    G, F, x0 and the step counter k.  Stepped with ``plant_step``, it reproduces ``closed_loop`` (box QP, tau_E
    constant).  Returns a dict with u, U, inner_iters, qp_iters and status (2 if x or u is not finite)."""
    Af, Bf, C = o.model_callables(p)
    x = np.asarray(x, dtype=np.float64).ravel()
    wmarg, w_dep = p["w_marg"], p["w_dep"]
    Q = np.array([[p["q11"], p["q12"]], [p["q12"], p["q22"]]])
    r = np.array([p["r1"], p["r2"]])
    lb, ub = p["umin"], p["umax"]

    def r1f(z):
        return o.rho1(z, wmarg, profile.rho1_variant)

    if not state:                                                              # offline build :63-73
        Rho1 = np.full(N, r1f(x)); Rho2 = np.full(N, o.rho2(x)); Rho3 = np.full(N, o.rho3(x, w_dep))
        Phi, Gamma, Lambda = o.Rho_to_PhiGammaLambda(Rho1, Rho2, Rho3, Af, Bf, C, profile.gamma_index)
        G, F = o.hessian_grad(Phi, Gamma, Lambda, x, r, Q)
        state.update(Rho1=Rho1, Rho2=Rho2, Rho3=Rho3, Uold=np.ones(N), G=G, F=F, x0=x.copy(), k=0)   # :86 (D13)
    Rho1, Rho2, Rho3, Uold, G, F = (state[key] for key in ("Rho1", "Rho2", "Rho3", "Uold", "G", "F"))
    inner, qpit, status = 0, 0, 0
    U = np.full(N, np.nan)
    with np.errstate(all="ignore"):
        for it in range(1, i_sim + 1):                                         # :94
            U, nit, st = qp(G, F, lb, ub)                                      # :97
            status = max(status, st)
            qpit += nit
            xN = np.zeros((2, N + 1)); xN[:, 0] = x                            # :110
            for i in range(N):                                                 # :112-117
                xN[:, i + 1] = Af(Rho1[i], Rho2[i]) @ xN[:, i] + Bf(Rho3[i]) * U[i] + C
                Rho1[i] = r1f(xN[:, i]); Rho2[i] = o.rho2(xN[:, i]); Rho3[i] = o.rho3(xN[:, i], w_dep)
            Phi, Gamma, Lambda = o.Rho_to_PhiGammaLambda(Rho1, Rho2, Rho3, Af, Bf, C, profile.gamma_index)  # :119
            xf = state["x0"] if profile.f_state == o.F_X0 else x
            G, F = o.hessian_grad(Phi, Gamma, Lambda, xf, r, Q)                  # :120-121
            inner = it
            if profile.inner_policy == o.INNER_EPS_BREAK and np.sum(np.abs(Uold - U)) < eps:   # :123
                break
            Uold = U.copy()                                                    # :127
    state.update(Uold=Uold, G=G, F=F, k=state["k"] + 1)
    u = float(U[0])                                                            # :107
    if not (np.all(np.isfinite(x)) and np.isfinite(u)):
        status = max(status, 2)
    return dict(u=u, U=U.copy(), inner_iters=inner, qp_iters=qpit, status=status)
