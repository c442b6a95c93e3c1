"""The perturbed loop with getWLc's state rows kept (ntm_mpc_closed_loop_perturbed_sc) without a GPU: its NumPy twin
(tests/perturbed_sc_oracle.py) is oracle.closed_loop(state_rows=...) when nothing is perturbed and the box-QP perturbed
twin with the rows off; the Python front end checks the new arguments before any library call, montecarlo.run takes
state rows together with a perturbation, and MEX gateway 12 rejects bad state-row arguments with ntm:arg."""
import dataclasses

import numpy as np
import pytest

from oracle import ntm_oracle as o
from perturbed_oracle import closed_loop_perturbed
from perturbed_sc_oracle import closed_loop_perturbed_sc

KEYS = ("xk", "uk", "Uk", "inner_iters", "qp_iters", "cost", "status")
XB = (0.05, 0.16, 2000.0, 12000.0)          # tests/test_controller_sc_cpu.py: binds on part of config 3, infeasible on another
GAMMA_I_FIXED = dataclasses.replace(o.LITERAL_FIXED, gamma_index=o.GAMMA_I)
GAMMA_I = dataclasses.replace(o.LITERAL, gamma_index=o.GAMMA_I)

CASES = [(mode, prof) for mode in (o.STATE_ROWS_REFRESH, o.STATE_ROWS_FROZEN)
         for prof in (o.LITERAL_FIXED, o.LITERAL, GAMMA_I_FIXED, GAMMA_I)]


@pytest.mark.parametrize("mode,profile", CASES,
                         ids=[f"{'refresh' if m == 1 else 'frozen'}-{'gamma_i' if p.gamma_index == o.GAMMA_I else 'literal'}-"
                              f"{'fixed' if p.inner_policy == o.INNER_FIXED else 'eps_break'}" for m, p in CASES])
def test_unperturbed_twin_is_the_state_row_closed_loop(mode, profile):
    N, k_sim, i_sim = 10, 8, 3
    phys, x0, _ = o.make_batch(3, S=40)
    n_inf = n_ok = 0
    for s in (0, 1, 2, 8, 28, 36):                 # XB: 8 starts outside the box, 28 and 36 leave it at steps 5 and 3
        p = o.scenario(phys, s)
        ref = o.closed_loop(p, x0[s], N=N, k_sim=k_sim, i_sim=i_sim, profile=profile, state_rows=mode, xbounds=XB)
        got = closed_loop_perturbed_sc(p, x0[s], N=N, k_sim=k_sim, i_sim=i_sim, profile=profile, state_rows=mode,
                                       xbounds=XB)
        for key in KEYS:
            assert np.array_equal(got[key], ref[key], equal_nan=True), (s, key)
        n_ok += ref["status"] == 0
        n_inf += got["k_inf"] is not None
    assert n_ok >= 1 and n_inf >= 2, (n_ok, n_inf)


def _perturbed_case(seed=3):
    phys, x0, _ = o.make_batch(2, S=8)
    p = o.scenario(phys, 5)
    pp = dict(p, Cw=p["Cw"] * 1.7, c_tauE=0.8)          # a plant the controller does not know
    rng = np.random.default_rng(seed)
    k_sim = 12
    d = rng.normal(size=(k_sim, 2)) * np.array([2e-3, 50.0])
    v = rng.normal(size=(k_sim, 2)) * np.array([1e-3, 20.0])
    return p, pp, x0[5], k_sim, d, v


@pytest.mark.parametrize("plant_profile", [o.LITERAL, dataclasses.replace(o.LITERAL, plant_integrator=o.PLANT_RK4),
                                           dataclasses.replace(o.LITERAL, tau_e_model=o.TAUE_W, plant_affine=o.PLANT_WITH_C)],
                         ids=["euler", "rk4", "taue_w_with_c"])
def test_rows_off_twin_is_the_box_qp_perturbed_twin(plant_profile):
    p, pp, x0, k_sim, d, v = _perturbed_case()
    ref = closed_loop_perturbed(p, x0, N=10, k_sim=k_sim, plant_p=pp, plant_profile=plant_profile, d=d, v=v)
    got = closed_loop_perturbed_sc(p, x0, N=10, k_sim=k_sim, state_rows=o.STATE_ROWS_OFF, plant_p=pp,
                                   plant_profile=plant_profile, d=d, v=v)
    for key in KEYS:
        assert np.array_equal(got[key], ref[key]), key


def test_noise_alone_makes_a_qp_infeasible():
    # the x_0 block of getWLc.m:30 tests y_k: a true state inside the box with a measurement outside it ends the run
    phys, x0, _ = o.make_batch(3, S=3)
    p = o.scenario(phys, 0)
    k_sim = 6
    clean = closed_loop_perturbed_sc(p, x0[0], N=10, k_sim=k_sim, i_sim=3, xbounds=XB)
    assert clean["k_inf"] is None
    v = np.zeros((k_sim, 2)); v[3, 0] = XB[1] - clean["xk"][0, 3] + 1e-3
    got = closed_loop_perturbed_sc(p, x0[0], N=10, k_sim=k_sim, i_sim=3, xbounds=XB, v=v)
    assert got["k_inf"] == 3 and got["status"] == o.QP_INFEASIBLE and np.isnan(got["cost"])
    assert np.array_equal(got["xk"][:, :4], clean["xk"][:, :4])
    assert np.all(np.isnan(got["xk"][:, 4:])) and np.all(np.isnan(got["uk"][3:]))
    assert np.all(got["inner_iters"][4:] == 0) and got["inner_iters"][3] > 0


def test_python_argument_checks():
    from ntm_mpc.api import MC_STATE_BOX, state_box_inputs
    assert state_box_inputs(0, None) is None
    assert np.array_equal(state_box_inputs(1, None), np.asarray(MC_STATE_BOX, dtype=np.float64))
    assert np.array_equal(state_box_inputs(2, XB), np.array(XB))
    bad = [
        ((3, None), "state_rows must be"),
        ((-1, None), "state_rows must be"),
        ((1, (0.1, 0.05, 2000.0, 12000.0)), "xmin > xmax"),
        ((2, (0.05, 0.16, np.nan, 12000.0)), "xmin > xmax"),
        ((1, (0.05, 0.16, 2000.0)), "xbounds must be"),
    ]
    for args, msg in bad:
        with pytest.raises(ValueError, match=msg):
            state_box_inputs(*args)


@pytest.mark.filterwarnings("ignore::RuntimeWarning")        # the recorder leaves the statistics buffer unwritten
def test_montecarlo_routes_state_rows_with_a_perturbation(monkeypatch):
    """montecarlo.run with state rows AND a perturbed plant calls the perturbed entry with the rows and the box (the
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
    box = (0.05, 0.16, 2000.0, 12000.0)
    res = montecarlo.run(3, S=16, k_sim=4, handle=h, state_rows=2, bounds=box, plant_sample={"Cw": (0.5, 2.0)},
                         w_std=(1e-3, 10.0), v_std=(1e-3, 10.0))
    names = [c[0] for c in h.calls]
    assert "closed_loop_perturbed_dev" in names and "closed_loop_sc_dev" not in names, names
    _, args, kw = h.calls[names.index("closed_loop_perturbed_dev")]
    assert kw["state_rows"] == 2 and tuple(kw["xbounds"]) == box
    assert args[10] != 0 and args[13] != 0 and args[14] != 0   # plant block, d and v all passed
    assert res["state_rows"] == 2


def test_mex_perturbed_gateway_rejects_bad_state_row_arguments():
    from test_mex_gateway import Mock
    mock = Mock()
    mock.workspace({})
    N, S, k_sim = 3, 2, 4
    x = np.array([[0.08, 0.1], [6000.0, 7000.0]])
    P = np.tile(o.derive_params(o.default_physics())[:, None], (1, S))
    E = np.zeros((0, 0))
    lo, hi = np.array([0.05, 2000.0]), np.array([0.16, 12000.0])
    base = [x, P, N, k_sim, 10, 1e-14, 0, E, 0, E, E]
    bad = [
        (base + [1], "usage"),                                    # 12 arguments
        (base + [1, lo], "usage"),                                # 13 arguments
        (base + [3, lo, hi], "state_rows must be"),
        (base + [-1, lo, hi], "state_rows must be"),
        (base + [1, hi, lo], "xmin must be <= xmax"),
        (base + [1, lo[:1], hi], "xmin and xmax"),
        ([x, P, 40, k_sim, 10, 1e-14, 2, E, 0, E, E, 1, lo, hi], "N <= 32"),   # GAMMA_I rows beyond one warp
    ]
    for args, msg in bad:
        with pytest.raises(RuntimeError, match=msg) as ei:
            mock.call("ntm_mpc_batch_perturbed", args, nlhs=5)
        assert str(ei.value).startswith("ntm:arg:"), str(ei.value)
