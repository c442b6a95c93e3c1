"""The receding-horizon controller step (ntm_mpc_step) without a GPU: the NumPy restatement of one step
(tests/controller_oracle.py) stepped with oracle.plant_step IS oracle.closed_loop, the record size of the header agrees
with the Python mirror, and MEX gateway 11 rejects bad calls before it touches the GPU."""
import dataclasses
import os
import re

import numpy as np
import pytest

from controller_oracle import controller_step
from oracle import ntm_oracle as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def stepped(p, x0, N, k_sim=20, i_sim=10, eps=1e-14, profile=o.LITERAL):
    state, x = {}, np.asarray(x0, dtype=np.float64).copy()
    xk, uk, Uk, inner, qpit, status = [x], [], [], [], [], 0
    for _ in range(k_sim):
        r = controller_step(p, state, x, N, i_sim, eps, profile)
        x = o.plant_step(p, x, r["u"], profile)
        xk.append(x); uk.append(r["u"]); Uk.append(r["U"])
        inner.append(r["inner_iters"]); qpit.append(r["qp_iters"]); status = max(status, r["status"])
    return dict(xk=np.array(xk).T, uk=np.array(uk), Uk=np.array(Uk).T, inner_iters=np.array(inner, dtype=np.int32),
                qp_iters=np.array(qpit, dtype=np.int32), status=status)


CASES = [
    ("default_fixed", 1, 0, 3, o.LITERAL_FIXED),
    ("default_eps_break", 1, 0, 3, o.LITERAL),
    ("config2_sample", 2, 17, 10, o.LITERAL),
    ("consistent", 2, 5, 10, o.CONSISTENT),
    ("f_xk_alone", 2, 9, 10, dataclasses.replace(o.LITERAL, f_state=o.F_XK)),
]


@pytest.mark.parametrize("name,cfg,s,N,profile", CASES, ids=[c[0] for c in CASES])
def test_controller_step_with_plant_step_is_the_closed_loop(name, cfg, s, N, profile):
    phys, x0, _ = o.make_batch(cfg, S=s + 1)
    p = o.scenario(phys, s)
    ref = o.closed_loop(p, x0[s], N=N, profile=profile)
    got = stepped(p, x0[s], N, profile=profile)
    for key in ("xk", "uk", "Uk", "inner_iters", "qp_iters"):
        assert np.array_equal(got[key], ref[key]), key
    assert got["status"] == ref["status"]
    r = np.array([p["r1"], p["r2"]]); Q = np.array([[p["q11"], p["q12"]], [p["q12"], p["q22"]]])
    e = got["xk"][:, 1:] - r[:, None]
    assert float(np.sum(e * (Q @ e))) == pytest.approx(ref["cost"], rel=1e-14)


def test_a_fresh_state_dict_restarts_the_controller():
    p = o.default_physics()
    a, b = {}, {}
    for _ in range(3):
        controller_step(p, a, o.default_x0(), 3)
    ra = controller_step(p, {}, o.default_x0(), 3)
    rb = controller_step(p, b, o.default_x0(), 3)
    assert np.array_equal(ra["U"], rb["U"]) and ra["inner_iters"] == rb["inner_iters"] and b["k"] == 1 and a["k"] == 3


def test_ctrl_doubles_matches_the_header():
    import ntm_mpc
    with open(os.path.join(ROOT, "include", "ntm_mpc.h")) as f:
        m = re.search(r"#define\s+NTM_CTRL_DOUBLES\(N\)\s+(.+)", f.read())
    assert m, "NTM_CTRL_DOUBLES not defined"
    expr = m.group(1).split("/*")[0].strip()
    for N in (1, 20, 32, 33, 100, 128):
        assert eval(expr, {"N": N}) == ntm_mpc.ctrl_doubles(N), N


def test_mex_step_gateway_rejects_bad_calls_before_touching_the_gpu():
    from test_mex_gateway import Mock
    mock = Mock()
    mock.workspace({})
    N, S = 3, 2
    ld = 7 * N + 7
    x = np.array([[0.08, 0.1], [6000.0, 7000.0]])
    P = np.tile(o.derive_params(o.default_physics())[:, None], (1, S))
    E = np.zeros((0, 0))
    bad = [
        ([E, x, P, N, 10, 1e-14], "usage"),                                     # wrong nrhs
        ([E, np.zeros((3, S)), P, N, 10, 1e-14, 0], "2 x S"),                   # x not 2 x S
        ([np.zeros((ld + 1, S)), x, P, N, 10, 1e-14, 0], "7N\\+7 rows"),         # state rows != NTM_CTRL_DOUBLES(N)
        ([np.zeros((ld, S + 1)), x, P, N, 10, 1e-14, 0], "7N\\+7 rows"),         # state columns != S
        ([E, x, np.zeros((15, 1)), N, 10, 1e-14, 0], "16 x 1"),                 # params not 16 x 1 / 16 x S
        ([E, x, np.zeros((16, 3)), N, 10, 1e-14, 0], "16 x 1"),
        ([E, x, P, 0, 10, 1e-14, 0], "N in 1..128"),
        ([E, x, P, 129, 10, 1e-14, 0], "N in 1..128"),
        ([E, x, P, N, 10, 1e-14, 128], "TAUE_W"),                               # profile bit 128
    ]
    for args, msg in bad:
        with pytest.raises(RuntimeError, match=msg) as ei:
            mock.call("ntm_mpc_step", args, nlhs=2)
        assert str(ei.value).startswith("ntm:arg:"), str(ei.value)
