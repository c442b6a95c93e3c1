"""The state observer (ntm_kf_step, ntm_mpc_closed_loop_observed) without a GPU: its NumPy twin (tests/observer_oracle.py)
is oracle.closed_loop (box QP and state rows) when nothing is perturbed, and the filter step is the textbook Kalman
recursion when rho is frozen; the Python front end, montecarlo.run and MEX gateways 12 and 13 check the new arguments
before any library call; the new symbols are exported."""
import dataclasses
import os
import re

import numpy as np
import pytest

from oracle import ntm_oracle as o
from observer_oracle import closed_loop_observed, kf_step

KEYS = ("xk", "uk", "Uk", "inner_iters", "qp_iters", "cost", "status")
XB = (0.05, 0.16, 2000.0, 12000.0)          # binds on part of config 3 and is infeasible on another
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RK4_C = dataclasses.replace(o.LITERAL_FIXED, plant_integrator=o.PLANT_RK4, plant_affine=o.PLANT_WITH_C)
GAMMA_I = dataclasses.replace(o.LITERAL, gamma_index=o.GAMMA_I)


def random_kf_cov(rng):
    """A valid kf_cov with correlated components: Qw PSD (here rank one), Rv PD."""
    a = rng.normal(size=2) * np.array([1e-3, 30.0])
    L = np.array([[5e-4, 0.0], [rng.normal() * 5.0, 20.0]])
    Q = np.outer(a, a); R = L @ L.T
    return np.array([Q[0, 0], Q[1, 0], Q[1, 1], R[0, 0], R[1, 0], R[1, 1]])


CASES = [(mode, prof) for mode in (o.STATE_ROWS_OFF, o.STATE_ROWS_REFRESH, o.STATE_ROWS_FROZEN)
         for prof in (o.LITERAL_FIXED, GAMMA_I, RK4_C)]


@pytest.mark.parametrize("mode,profile", CASES, ids=[f"rows{m}-{i}" for i, (m, _) in enumerate(CASES)])
def test_unperturbed_twin_is_the_closed_loop(mode, profile):
    """Nothing perturbed: the filter's prediction is the plant itself, the innovation is exactly zero and xhat = x, so
    the observed loop is oracle.closed_loop bit for bit, whatever the covariances."""
    N, k_sim, i_sim = 10, 8, 3
    phys, x0, _ = o.make_batch(3, S=40)
    rng = np.random.default_rng(1)
    n_inf = 0
    for s in (0, 1, 8, 28, 36):                 # XB: 8 starts outside the box, 28 and 36 leave it later
        p = o.scenario(phys, s)
        kw = dict(state_rows=mode, xbounds=XB) if mode else {}
        ref = o.closed_loop(p, x0[s], N=N, k_sim=k_sim, i_sim=i_sim, profile=profile, **kw)
        got = closed_loop_observed(p, x0[s], N=N, k_sim=k_sim, i_sim=i_sim, profile=profile, state_rows=mode,
                                   xbounds=XB, kf_cov=random_kf_cov(rng))
        for key in KEYS:
            assert np.array_equal(got[key], ref[key], equal_nan=True), (s, key)
        live = np.isfinite(got["xhat"][0])
        assert np.array_equal(got["xhat"][:, live], ref["xk"][:, :k_sim][:, live])
        if got["k_inf"] is not None:
            n_inf += 1
            assert np.all(np.isnan(got["xhat"][:, got["k_inf"] + 1:]))
            assert np.array_equal(got["xhat"][:, got["k_inf"]], ref["xk"][:, got["k_inf"]])
    assert (n_inf >= 1) == (mode != o.STATE_ROWS_OFF), n_inf


def test_frozen_rho_filter_is_the_textbook_kalman_recursion(monkeypatch):
    """rho frozen at one point: the model is linear, x+ = A x + B u (+ C), and the twin's step must be the textbook
    recursion (P- = A P A' + Q, K = P- (P- + R)^-1, standard-form update), whose covariance converges to the solution
    of the discrete algebraic Riccati equation.  P stays symmetric with det >= 0."""
    from scipy.linalg import solve_discrete_are
    p = o.default_physics()
    xs = np.array([0.08, 6000.0])
    r1, r2, r3 = o.rho1(xs, p["w_marg"]), o.rho2(xs), o.rho3(xs, p["w_dep"])
    monkeypatch.setattr(o, "rho1", lambda x, wmarg, variant=0: r1)
    monkeypatch.setattr(o, "rho2", lambda x: r2)
    monkeypatch.setattr(o, "rho3", lambda x, w_dep: r3)
    Af, Bf, C = o.model_callables(p)
    A, B = Af(r1, r2), Bf(r3)
    prof = dataclasses.replace(o.LITERAL, plant_affine=o.PLANT_WITH_C)
    kc = np.array([1e-6, 2e-3, 900.0, 2.5e-7, -1e-3, 400.0])
    Q = np.array([[kc[0], kc[1]], [kc[1], kc[2]]]); R = np.array([[kc[3], kc[4]], [kc[4], kc[5]]])
    rng = np.random.default_rng(7)
    rec = np.zeros(6)
    xh, P = None, None
    for k in range(60):
        y = xs + rng.normal(size=2) * np.array([5e-4, 20.0])
        u = 1e5 * (1 + k % 3)
        rec = kf_step(p, rec, y, u, kc, prof)
        if k == 0:
            xh, P = y.copy(), R.copy()
        else:
            xm = A @ xh + B * u + C
            Pm = A @ P @ A.T + Q
            K = np.linalg.solve((Pm + R).T, Pm.T).T
            xh = xm + K @ (y - xm)
            P = (np.eye(2) - K) @ Pm
            P = 0.5 * (P + P.T)
        Pt = np.array([[rec[2], rec[3]], [rec[3], rec[4]]])
        assert np.allclose(rec[:2], xh, rtol=1e-12, atol=0), k
        scale = np.sqrt(np.outer(np.diag(P), np.diag(P)))
        assert np.all(np.abs(Pt - P) <= 1e-9 * scale), k
        assert rec[2] >= 0 and rec[4] >= 0 and rec[2] * rec[4] - rec[3] ** 2 >= 0, k
        assert rec[5] == k + 1
    Pinf = solve_discrete_are(A.T, np.eye(2), Q, R)        # the steady-state prior covariance
    Pm = A @ Pt @ A.T + Q
    assert np.allclose(Pm, Pinf, rtol=1e-6, atol=0)


def test_fresh_record_takes_the_measurement():
    p = o.default_physics()
    kc = (1e-6, 0.0, 900.0, 2.5e-7, 0.0, 400.0)
    rec = kf_step(p, np.zeros(6), [0.07, 5000.0], np.nan, kc)             # u is not read
    assert np.array_equal(rec, [0.07, 5000.0, 2.5e-7, 0.0, 400.0, 1.0])


def test_python_argument_checks():
    import ntm_mpc
    from ntm_mpc.api import NtmMpc, Observer, kf_cov_input
    good = (1e-6, 0.0, 900.0, 2.5e-7, 0.0, 400.0)
    assert np.array_equal(kf_cov_input(good), np.array(good))
    assert np.array_equal(kf_cov_input((0.0, 0.0, 0.0, 1.0, 0.5, 1.0)), [0.0, 0.0, 0.0, 1.0, 0.5, 1.0])
    bad = [
        (None, "kf_cov is required"),
        ((1.0, 0.0, 1.0, 1.0, 0.0), "6 entries"),
        ((1.0, 0.0, np.nan, 1.0, 0.0, 1.0), "non-finite"),
        ((1.0, 0.0, 1.0, np.inf, 0.0, 1.0), "non-finite"),
        ((-1e-9, 0.0, 1.0, 1.0, 0.0, 1.0), "Qw is not positive semi-definite"),
        ((1.0, 2.0, 1.0, 1.0, 0.0, 1.0), "Qw is not positive semi-definite"),
        ((1.0, 0.0, 1.0, 0.0, 0.0, 1.0), "Rv is not positive definite"),
        ((1.0, 0.0, 1.0, 1.0, 1.0, 1.0), "Rv is not positive definite"),
    ]
    for c, msg in bad:
        with pytest.raises(ValueError, match=msg):
            kf_cov_input(c)
    # the front end refuses a bad record or covariance before the library is called (no handle needed)
    h = object.__new__(NtmMpc)
    P = o.derive_params(o.default_physics())
    y = np.array([[0.08, 6000.0], [0.09, 6100.0]])
    for state in (np.zeros((2, 7)), np.zeros((3, 6)), np.zeros((2, 6), dtype=np.float32), np.zeros((6, 2)).T):
        with pytest.raises(ValueError, match="state must be"):
            h.kf_step(state, y, [0.0, 0.0], P, good)
    with pytest.raises(ValueError, match="Rv"):
        h.kf_step(np.zeros((2, 6)), y, [0.0, 0.0], P, (1.0, 0.0, 1.0, 0.0, 0.0, 1.0))
    with pytest.raises(ValueError, match="Qw"):
        Observer(h, P, (1.0, 3.0, 1.0, 1.0, 0.0, 1.0), S=2)
    with pytest.raises(ValueError, match="S is needed"):
        Observer(h, P, good)
    obs = Observer(h, np.tile(P, (3, 1)), good)
    assert obs.state.shape == (3, ntm_mpc.kf_doubles()) and obs.S == 3
    obs.state[:] = 1.0
    obs.reset([False, True, False])
    assert np.all(obs.state[1] == 0.0) and np.all(obs.state[[0, 2]] == 1.0)
    obs.reset()
    assert np.all(obs.state == 0.0)
    with pytest.raises(ValueError, match="kf_cov is required"):
        h.closed_loop_observed(y, P, 10, None)


def test_new_symbols_are_exported():
    import ntm_mpc
    from ntm_mpc import _lib, montecarlo
    assert ntm_mpc.kf_doubles() == 6
    for name in ("Observer", "kf_cov_input", "kf_doubles"):
        assert hasattr(ntm_mpc, name), name
    assert callable(montecarlo.kf_cov_from_std)
    for name in ("ntm_kf_step", "ntm_kf_step_dev", "ntm_mpc_closed_loop_observed", "ntm_mpc_closed_loop_observed_dev"):
        assert name in _lib.SYMBOLS, name
    hdr = open(os.path.join(ROOT, "include", "ntm_mpc.h")).read()
    assert re.search(r"#define NTM_KF_DOUBLES 6\b", hdr)
    for name in ("ntm_kf_step", "ntm_kf_step_dev", "ntm_mpc_closed_loop_observed", "ntm_mpc_closed_loop_observed_dev"):
        m = re.search(r"int %s\(([^;]*)\);" % name, hdr)
        assert m, name
        assert len(m.group(1).split(",")) == len(_lib.SYMBOLS[name][1]), name
    nm = os.path.join(ROOT, "mpc-ntm-control_b200", "lib", "libntm_mpc.so")
    if os.path.exists(nm):
        import ctypes
        lib = ctypes.CDLL(nm)
        for name in ("ntm_kf_step", "ntm_kf_step_dev", "ntm_mpc_closed_loop_observed", "ntm_mpc_closed_loop_observed_dev"):
            assert hasattr(lib, name), name


def test_kf_cov_from_std():
    from ntm_mpc import montecarlo
    c = montecarlo.kf_cov_from_std((1e-3, 30.0), (5e-4, 20.0))
    assert np.allclose(c, [1e-6, 0.0, 900.0, 2.5e-7, 0.0, 400.0], rtol=1e-15, atol=0)
    assert np.allclose(montecarlo.kf_cov_from_std(None, 2.0), [0.0, 0.0, 0.0, 4.0, 0.0, 4.0])
    with pytest.raises(ValueError, match="v_std is required"):
        montecarlo.kf_cov_from_std(1.0, None)
    with pytest.raises(ValueError, match="Rv"):
        montecarlo.kf_cov_from_std(1.0, (0.0, 1.0))


@pytest.mark.filterwarnings("ignore::RuntimeWarning")        # the recorder leaves the statistics buffer unwritten
def test_montecarlo_routes_kf_cov_to_the_observed_entry(monkeypatch):
    """montecarlo.run(kf_cov=...) calls the observed entry with the plant, the noise, the rows and the covariances (the
    device buffers live on the CPU here: the handle is a recorder)."""
    import torch
    from ntm_mpc import montecarlo
    real_device = torch.device
    monkeypatch.setattr(torch, "device", lambda *a, **k: real_device("cpu"))
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: type("St", (), {"cuda_stream": 0})())

    class Recorder:
        def __init__(self):
            self.calls = []

        def __getattr__(self, name):
            return lambda *a, **k: self.calls.append((name, a, k))

    h = Recorder()
    kc = montecarlo.kf_cov_from_std((1e-3, 30.0), (5e-4, 20.0))
    res = montecarlo.run(3, S=16, k_sim=4, handle=h, state_rows=1, bounds=XB, plant_sample={"Cw": (0.5, 2.0)},
                         w_std=(1e-3, 30.0), v_std=(5e-4, 20.0), kf_cov=kc, trajectories=True)
    names = [c[0] for c in h.calls]
    assert "closed_loop_observed_dev" in names and "closed_loop_perturbed_dev" not in names, names
    _, args, kw = h.calls[names.index("closed_loop_observed_dev")]
    assert kw["state_rows"] == 1 and tuple(kw["xbounds"]) == XB and np.array_equal(kw["kf_cov"], kc)
    assert kw["xhat_ptr"] != 0
    assert args[10] != 0 and args[13] != 0 and args[14] != 0
    assert res["xhat"].shape == (16, 4, 2) and np.array_equal(res["kf_cov"], kc)
    with pytest.raises(ValueError, match="Rv"):
        montecarlo.run(3, S=16, k_sim=4, handle=Recorder(), kf_cov=(1.0, 0.0, 1.0, 0.0, 0.0, 1.0))


def test_mex_gateways_12_and_13_reject_bad_observer_arguments():
    from test_mex_gateway import Mock
    mock = Mock()
    mock.workspace({})
    N, S, k_sim = 3, 2, 4
    x = np.array([[0.08, 0.1], [6000.0, 7000.0]])
    P = np.tile(o.derive_params(o.default_physics())[:, None], (1, S))
    E = np.zeros((0, 0))
    lo, hi = np.array([0.05, 2000.0]), np.array([0.16, 12000.0])
    kc = np.array([1e-6, 0.0, 900.0, 2.5e-7, 0.0, 400.0])
    base = [x, P, N, k_sim, 10, 1e-14, 0, E, 0, E, E, 1, lo, hi]
    bad12 = [
        (base + [kc[:5]], "kf_cov must be"),
        (base + [np.array([1e-6, 0.0, np.nan, 2.5e-7, 0.0, 400.0])], "non-finite"),
        (base + [np.array([-1.0, 0.0, 900.0, 2.5e-7, 0.0, 400.0])], "Qw"),
        (base + [np.array([1e-6, 0.0, 900.0, 2.5e-7, 1.0, 400.0])], "Rv"),
        (base + [kc, 1.0], "usage"),                                          # 16 arguments
    ]
    for args, msg in bad12:
        with pytest.raises(RuntimeError, match=msg) as ei:
            mock.call("ntm_mpc_batch_perturbed", args, nlhs=6)
        assert str(ei.value).startswith("ntm:arg:"), str(ei.value)
    with pytest.raises(RuntimeError, match="needs the kf_cov") as ei:       # xhat without an observer
        mock.call("ntm_mpc_batch_perturbed", base, nlhs=6)
    assert str(ei.value).startswith("ntm:arg:")
    u = np.zeros((1, S))
    bad13 = [
        ([x, u, P, kc, E], "usage"),
        ([x, np.zeros((1, 3)), P, kc, E, 0], "u must be"),
        ([x, u, P[:5], kc, E, 0], "16 x 1"),
        ([x, u, P, kc[:4], E, 0], "kf_cov must be"),
        ([x, u, P, np.array([1e-6, 0.0, 900.0, 0.0, 0.0, 400.0]), E, 0], "Rv"),
        ([x, u, P, np.array([1e-6, 1.0, 900.0, 2.5e-7, 0.0, 400.0]), E, 0], "Qw"),
        ([x, u, P, kc, np.zeros((7, S)), 0], "6 rows by S"),
        ([x, u, P, kc, np.zeros((6, S + 1)), 0], "6 rows by S"),
        ([x, u, P, kc, E, 128], "TAUE_W"),
    ]
    for args, msg in bad13:
        with pytest.raises(RuntimeError, match=msg) as ei:
            mock.call("ntm_kf_step", args, nlhs=2)
        assert str(ei.value).startswith("ntm:arg:"), str(ei.value)
