"""The fused loop against a perturbed plant (ntm_mpc_closed_loop_perturbed) without a GPU: its NumPy twin
(tests/perturbed_oracle.py) is oracle.closed_loop when nothing is perturbed and the step-API composition when
something is, the Python front end checks its arguments before any library call, and MEX gateway 12 rejects bad
calls with ntm:arg."""
import dataclasses

import numpy as np
import pytest

from controller_oracle import controller_step
from oracle import ntm_oracle as o
from perturbed_oracle import closed_loop_perturbed

KEYS = ("xk", "uk", "Uk", "inner_iters", "qp_iters", "cost", "status")

CASES = [
    ("literal_fixed", 1, 0, 3, o.LITERAL_FIXED),
    ("literal_eps_break", 2, 17, 10, o.LITERAL),
    ("consistent_eps_break", 2, 5, 10, o.CONSISTENT),
    ("consistent_fixed", 2, 9, 10, o.CONSISTENT_FIXED),
]


@pytest.mark.parametrize("name,cfg,s,N,profile", CASES, ids=[c[0] for c in CASES])
def test_unperturbed_twin_is_the_closed_loop(name, cfg, s, N, profile):
    phys, x0, _ = o.make_batch(cfg, S=s + 1)
    p = o.scenario(phys, s)
    ref = o.closed_loop(p, x0[s], N=N, profile=profile)
    got = closed_loop_perturbed(p, x0[s], N=N, profile=profile)
    for key in KEYS:
        assert np.array_equal(got[key], ref[key]), key


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
def test_perturbed_twin_is_the_step_composition(plant_profile):
    p, pp, x0, k_sim, d, v = _perturbed_case()
    got = closed_loop_perturbed(p, x0, N=10, k_sim=k_sim, profile=o.LITERAL, plant_p=pp, plant_profile=plant_profile,
                                d=d, v=v)
    # written out: the controller sees x + v (v_0 included: its offline build runs from y_0), the plant is the oracle's
    # plant step on the plant's own physics, d is one add after it, the cost is judged on the true states
    state, x, xs, us, status = {}, x0.copy(), [x0.copy()], [], 0
    for k in range(k_sim):
        r = controller_step(p, state, x + v[k], 10, 10, 1e-14, o.LITERAL)
        x = o.plant_step(pp, x, r["u"], plant_profile) + d[k]
        xs.append(x); us.append(r["u"]); status = max(status, r["status"])
    xs = np.array(xs).T
    assert np.array_equal(state["x0"], x0 + v[0])
    assert np.array_equal(got["xk"], xs) and np.array_equal(got["uk"], np.array(us)) and got["status"] == status
    rr = np.array([p["r1"], p["r2"]]); Q = np.array([[p["q11"], p["q12"]], [p["q12"], p["q22"]]])
    e = xs[:, 1:] - rr[:, None]
    assert got["cost"] == float(np.sum(e * (Q @ e)))
    # and the perturbation matters: the unperturbed loop takes other inputs
    assert not np.array_equal(got["uk"], o.closed_loop(p, x0, N=10, k_sim=k_sim)["uk"])


def test_nonfinite_measurement_is_flagged():
    p, pp, x0, k_sim, d, v = _perturbed_case()
    v = v.copy(); v[4, 1] = np.nan
    got = closed_loop_perturbed(p, x0, N=10, k_sim=k_sim, plant_p=pp, d=d, v=v)
    assert got["status"] == 2


def test_python_argument_checks():
    from ntm_mpc import PROFILE_PLANT_RK4, PROFILE_TAUE_W, perturbed_inputs
    from ntm_mpc import physics
    prm = physics.params_from_physics(physics.nominal())
    x0 = np.tile(physics.x0_default(), (3, 1))
    k_sim = 4
    ok = perturbed_inputs(x0, prm, None, None, None, None, k_sim, PROFILE_PLANT_RK4 | 4)
    assert ok[3] is None and ok[4] == 1 and ok[5] == PROFILE_PLANT_RK4      # plant bits of the controller profile
    w = np.zeros((3, k_sim, 2))
    assert perturbed_inputs(x0, prm, np.tile(prm, (3, 1)), PROFILE_TAUE_W, w, w, k_sim, 0)[4] == 3
    bad = [
        (dict(profile=PROFILE_TAUE_W), "TAUE_W"),
        (dict(plant_profile=2), "plant_profile"),
        (dict(plant_profile=4), "plant_profile"),
        (dict(w=np.zeros((3, k_sim + 1, 2))), "w must be"),
        (dict(v=np.zeros((2, k_sim, 2))), "v must be"),
        (dict(plant_params=np.zeros((2, prm.size))), "params must be"),
        (dict(plant_params=np.zeros(5)), "params must have"),
    ]
    for kw, msg in bad:
        args = dict(plant_params=None, plant_profile=None, w=None, v=None, profile=0)
        args.update(kw)
        with pytest.raises(ValueError, match=msg):
            perturbed_inputs(x0, prm, args["plant_params"], args["plant_profile"], args["w"], args["v"], k_sim,
                             args["profile"])


def test_mex_perturbed_gateway_rejects_bad_arguments():
    from test_mex_gateway import Mock
    mock = Mock()
    mock.workspace({})
    N, S, k_sim = 3, 2, 4
    x = np.array([[0.08, 0.1], [6000.0, 7000.0]])
    P = np.tile(o.derive_params(o.default_physics())[:, None], (1, S))
    E = np.zeros((0, 0))
    W = np.zeros((2, k_sim * S))
    bad = [
        ([x, P, N, k_sim, 10, 1e-14, 0, E, 0, E], "usage"),                     # 10 arguments
        ([x, P, N, k_sim, 10, 1e-14, 128, E, 0, E, E], "TAUE_W"),               # controller-side tau_E(w)
        ([x, P, N, k_sim, 10, 1e-14, 0, E, 2, E, E], "plant_profile"),          # GAMMA_I is no plant bit
        ([x, P, N, k_sim, 10, 1e-14, 0, P[:, :1][:5], 0, E, E], "plant_params"),
        ([x, P, N, k_sim, 10, 1e-14, 0, np.tile(P, (1, 2)), 0, E, E], "plant_params"),   # 16 x 2S
        ([x, P, N, k_sim, 10, 1e-14, 0, E, 0, W[:, :-1], E], "w and v"),
        ([x, P, N, k_sim, 10, 1e-14, 0, E, 0, E, np.zeros((2, 1))], "w and v"),
        ([x, P, 0, k_sim, 10, 1e-14, 0, E, 0, E, E], "N in 1..128"),
        ([x, P[:5], N, k_sim, 10, 1e-14, 0, E, 0, E, E], "params must be"),
    ]
    for args, msg in bad:
        with pytest.raises(RuntimeError, match=msg) as ei:
            mock.call("ntm_mpc_batch_perturbed", args, nlhs=5)
        assert str(ei.value).startswith("ntm:arg:"), str(ei.value)
