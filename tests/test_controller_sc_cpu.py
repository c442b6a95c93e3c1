"""The controller step with getWLc's state rows kept (ntm_mpc_step_sc) without a GPU: the NumPy twin
(tests/controller_sc_oracle.py) stepped with oracle.plant_step IS oracle.closed_loop(state_rows=...), up to and
including the step at which a scenario turns infeasible; and MEX gateway 11 rejects bad state-row arguments."""
import dataclasses

import numpy as np
import pytest

from controller_sc_oracle import controller_step_sc
from oracle import ntm_oracle as o

XB = (0.05, 0.16, 2000.0, 12000.0)          # tests/test_gpu_ext.py: binds on part of config 3, infeasible on another
GAMMA_I_FIXED = dataclasses.replace(o.LITERAL_FIXED, gamma_index=o.GAMMA_I)
GAMMA_I = dataclasses.replace(o.LITERAL, gamma_index=o.GAMMA_I)


def stepped_sc(p, x0, N, k_sim, i_sim, profile, mode, xb):
    """k_sim x (controller_step_sc + plant_step); a scenario whose step comes back infeasible ends there, as the script does
    (closed_loop's outputs from that step on: NaN, iteration counts 0)."""
    state, x = {}, np.asarray(x0, dtype=np.float64).copy()
    xk = np.full((2, k_sim + 1), np.nan); xk[:, 0] = x
    uk = np.full(k_sim, np.nan); Uk = np.full((N, k_sim), np.nan)
    inner = np.zeros(k_sim, dtype=np.int32); qpit = np.zeros(k_sim, dtype=np.int32)
    status = 0
    for k in range(k_sim):
        before = {key: (v.copy() if isinstance(v, np.ndarray) else v) for key, v in state.items()}
        r = controller_step_sc(p, state, x, N, i_sim, 1e-14, profile, state_rows=mode, xbounds=xb)
        inner[k], qpit[k] = r["inner_iters"], r["qp_iters"]
        status = max(status, r["status"])
        if r["status"] == o.QP_INFEASIBLE:
            assert np.isnan(r["u"]) and np.all(np.isnan(r["U"]))
            assert state.keys() == before.keys()                          # the record is left as it was
            for key, v in before.items():
                assert (np.array_equal(state[key], v) if isinstance(v, np.ndarray)
                        else all(np.array_equal(a, b) for a, b in zip(state[key], v)) if isinstance(v, tuple)
                        else state[key] == v), key
            return dict(xk=xk, uk=uk, Uk=Uk, inner_iters=inner, qp_iters=qpit, status=status, k_inf=k)
        uk[k] = r["u"]; Uk[:, k] = r["U"]
        x = o.plant_step(p, x, r["u"], profile)
        xk[:, k + 1] = x
    if not np.all(np.isfinite(xk)):
        status = max(status, 2)
    return dict(xk=xk, uk=uk, Uk=Uk, inner_iters=inner, qp_iters=qpit, status=status, k_inf=None)


CASES = [(mode, prof) for mode in (o.STATE_ROWS_REFRESH, o.STATE_ROWS_FROZEN)
         for prof in (o.LITERAL_FIXED, o.LITERAL, GAMMA_I_FIXED, GAMMA_I)]


@pytest.mark.parametrize("mode,profile", CASES,
                         ids=[f"{'refresh' if m == 1 else 'frozen'}-{'gamma_i' if p.gamma_index == o.GAMMA_I else 'literal'}-"
                              f"{'fixed' if p.inner_policy == o.INNER_FIXED else 'eps_break'}" for m, p in CASES])
def test_state_row_controller_step_with_plant_step_is_the_closed_loop(mode, profile):
    N, k_sim, i_sim = 10, 8, 3
    phys, x0, _ = o.make_batch(3, S=40)
    n_inf_first = n_inf_later = n_ok = 0
    for s in (0, 1, 2, 8, 28, 36):                 # XB: 8 starts outside the box, 28 and 36 leave it at steps 5 and 3
        p = o.scenario(phys, s)
        ref = o.closed_loop(p, x0[s], N=N, k_sim=k_sim, i_sim=i_sim, profile=profile, state_rows=mode, xbounds=XB)
        got = stepped_sc(p, x0[s], N, k_sim, i_sim, profile, mode, XB)
        for key in ("xk", "uk", "Uk", "inner_iters", "qp_iters"):
            assert np.array_equal(got[key], ref[key], equal_nan=True), (s, key)
        assert got["status"] == ref["status"], s
        n_ok += ref["status"] == 0
        n_inf_first += got["k_inf"] == 0
        n_inf_later += got["k_inf"] is not None and got["k_inf"] > 0
    # the sample has scenarios that run to the end, one infeasible on its first step (fresh record) and ones that turn
    # infeasible after feasible steps
    assert n_ok >= 1 and n_inf_first >= 1 and n_inf_later >= 2, (n_ok, n_inf_first, n_inf_later)


def test_frozen_rows_are_the_offline_build_and_stay():
    p, x, N = o.default_physics(), o.default_x0(), 3
    wide = (0.0, 1.0, 0.0, 1e9)
    fr = {}
    r0 = controller_step_sc(p, fr, x, N, state_rows=o.STATE_ROWS_FROZEN, xbounds=wide)
    rho = (np.full(N, o.rho1(x, p["w_marg"], o.LITERAL.rho1_variant)), np.full(N, o.rho2(x)), np.full(N, o.rho3(x, p["w_dep"])))
    offline = o.Rho_to_PhiGammaLambda(*rho, *o.model_callables(p), o.LITERAL.gamma_index)      # :63-66, :74
    rows0 = fr["rows"]
    assert all(np.array_equal(a, b) for a, b in zip(rows0, offline))
    x1 = o.plant_step(p, x, r0["u"], o.LITERAL)
    controller_step_sc(p, fr, x1, N, state_rows=o.STATE_ROWS_FROZEN, xbounds=wide)
    assert fr["k"] == 2 and all(a is b for a, b in zip(fr["rows"], rows0))


def test_mex_step_gateway_rejects_bad_state_row_arguments():
    from test_mex_gateway import Mock
    mock = Mock()
    mock.workspace({})
    N, S = 3, 2
    x = np.array([[0.08, 0.1], [6000.0, 7000.0]])
    P = np.tile(o.derive_params(o.default_physics())[:, None], (1, S))
    E = np.zeros((0, 0))
    lo, hi = np.array([0.05, 2000.0]), np.array([0.16, 12000.0])
    bad = [
        ([E, x, P, N, 10, 1e-14, 0, 1, lo], "usage"),                          # 9 arguments
        ([E, x, P, N, 10, 1e-14, 0, 3, lo, hi], "state_rows"),                 # unknown mode
        ([E, x, P, N, 10, 1e-14, 0, -1, lo, hi], "state_rows"),
        ([E, x, P, N, 10, 1e-14, 0, 1, lo[:1], hi], "2-vectors"),              # xmin not 2 x 1
        ([E, x, P, N, 10, 1e-14, 0, 1, lo, np.zeros(3)], "2-vectors"),
        ([E, x, P, N, 10, 1e-14, 0, 1, hi, lo], "xmin must be <= xmax"),       # inverted box
        ([E, x, P, N, 10, 1e-14, 0, 1, np.array([np.nan, 0.0]), hi], "xmin must be <= xmax"),
        ([E, x, P, 40, 10, 1e-14, 2, 1, lo, hi], "N <= 32"),                   # dense Gamma rows beyond N = 32
        ([E, x, P, N, 10, 1e-14, 128, 1, lo, hi], "TAUE_W"),
    ]
    for args, msg in bad:
        with pytest.raises(RuntimeError, match=msg) as ei:
            mock.call("ntm_mpc_step", args, nlhs=2)
        assert str(ei.value).startswith("ntm:arg:"), str(ei.value)
