"""The controller step with getWLc's state rows kept (ntm_mpc_step_sc[_dev]) on the GPU (-m gpu).

k_sim controller steps, each followed by ntm_plant_step under the same profile, must reproduce the fused state-row loop
(ntm_mpc_closed_loop_sc) bit for bit on every state-row instantiation: one warp with the literal Gamma (Toeplitz rows)
and the dense Gamma (N <= 32), and the multi-warp literal groups.  A scenario whose step comes back infeasible ends there,
as the script does; the harness then holds its measured state.  Then the infeasible-step contract, STATE_ROWS_OFF against
ntm_mpc_step, restarts with a new x0, a disturbed and noisy plant against the NumPy twin, the C ABI contract and MEX
gateway 11 against gateway 8."""

import os
import subprocess
import sys

import numpy as np
import pytest

from controller_sc_oracle import controller_step_sc
from oracle import ntm_oracle as o

pytestmark = pytest.mark.gpu

FIXED, GAMMA_I, DENSE_G, CONS = 16, 2, 32, 2 | 4 | 8
REFRESH, FROZEN = 1, 2
XB = (0.05, 0.16, 2000.0, 12000.0)          # tests/test_gpu_ext.py: binds on part of config 3, infeasible on another
SCRIPT_BOX = (0.06, 0.15, 100 * 2 * np.pi, 5000 * 2 * np.pi)   # NTM_MPC_Sim.m:39-45 (ntm_mpc.api.MC_STATE_BOX)
INFEASIBLE = 3


@pytest.fixture(scope="module")
def mpc():
    import ntm_mpc
    h = ntm_mpc.NtmMpc(0)
    yield h
    h.close()


def batch(S, N):
    phys, x0, _ = o.make_batch(3, S=S)
    return o.derive_params_batch(phys).T.copy(), x0, N


def end_at_infeasible(r):
    """The script cannot continue past an infeasible QP (:100-101): from the step after it on, everything is NaN / 0,
    as ntm_mpc_closed_loop_sc reports it."""
    st = r["step_status"]
    S, k_sim = st.shape
    for s in range(S):
        bad = np.flatnonzero(st[s] == INFEASIBLE)
        if bad.size:
            k = bad[0]
            r["xk"][s, k + 1:] = np.nan; r["uk"][s, k + 1:] = np.nan; r["Uk"][s, k + 1:] = np.nan
            r["inner_iters"][s, k + 1:] = 0; r["qp_iters"][s, k + 1:] = 0; st[s, k + 1:] = 0
    return r


def controller_run_sc(mpc, x0, P, N, mode, xb, k_sim=8, i_sim=3, eps=1e-14, profile=0, layout=0, host=False,
                      stream=None):
    """k_sim x (ntm_mpc_step_sc[_dev] + ntm_plant_step[_dev]); a scenario whose step is infeasible keeps its measured
    state (its record is unchanged, so every later call repeats the verdict).  Returns the fused loop's outputs."""
    import torch
    import ntm_mpc
    S = x0.shape[0]
    if host:
        state = np.zeros((S, ntm_mpc.ctrl_doubles(N)))
        x, out = x0.copy(), []
        for _ in range(k_sim):
            r = mpc.mpc_step(state, x, P, N, i_sim, eps, profile, want_U=True, state_rows=mode, xbounds=xb)
            out.append((x, r["u"], r["U"], r["inner_iters"], r["qp_iters"], r["status"]))
            xn = mpc.plant_step(x, r["u"], P, profile)
            dead = r["status"] == INFEASIBLE
            xn[dead] = x[dead]
            x = xn
        xs = [t[0] for t in out] + [x]
        return end_at_infeasible(dict(
            xk=np.stack(xs, 1), uk=np.stack([t[1] for t in out], 1), Uk=np.stack([t[2] for t in out], 1),
            inner_iters=np.stack([t[3] for t in out], 1), qp_iters=np.stack([t[4] for t in out], 1),
            step_status=np.stack([t[5] for t in out], 1)))
    dev = torch.device("cuda")
    soa = layout == ntm_mpc.LAYOUT_SOA
    x = torch.tensor(x0.T.copy() if soa else x0, device=dev)
    p = torch.tensor(P.T.copy() if soa else P, device=dev)
    state = torch.zeros(S, ntm_mpc.ctrl_doubles(N), dtype=torch.float64, device=dev)
    u = torch.empty(S, dtype=torch.float64, device=dev)
    U = torch.empty((N, S) if soa else (S, N), dtype=torch.float64, device=dev)
    it = torch.empty((3, S), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    if stream is not None:
        mpc.set_stream(stream.cuda_stream)
    hist = []
    for _ in range(k_sim):
        mpc.mpc_step_dev(S, N, i_sim, eps, profile, layout, x.data_ptr(), p.data_ptr(), S, state.data_ptr(), u.data_ptr(),
                         U.data_ptr(), it[0].data_ptr(), it[1].data_ptr(), it[2].data_ptr(), state_rows=mode, xbounds=xb)
        xn = torch.empty_like(x)
        mpc.plant_step_dev(S, profile, layout, x.data_ptr(), u.data_ptr(), p.data_ptr(), S, xn.data_ptr())
        if stream is None:
            mpc.sync()
        hist.append((x, u.clone(), U.clone(), it.clone()))           # on the caller's stream: ordered, no host sync
        dead = it[2] == INFEASIBLE
        xn = torch.where(dead[None, :] if soa else dead[:, None], x, xn)
        if stream is None:
            torch.cuda.current_stream().synchronize()                # the copies are done before the next step writes
        x = xn
    if stream is not None:
        mpc.reset_stream()
    torch.cuda.synchronize()
    mpc.sync()
    cpu = lambda t: t.cpu().numpy()
    xs = [cpu(h[0]) for h in hist] + [cpu(x)]
    if soa:
        xs = [a.T for a in xs]
    Us = [cpu(h[2]).T if soa else cpu(h[2]) for h in hist]
    its = [cpu(h[3]) for h in hist]
    return end_at_infeasible(dict(
        xk=np.stack(xs, 1), uk=np.stack([cpu(h[1]) for h in hist], 1), Uk=np.stack(Us, 1),
        inner_iters=np.stack([a[0] for a in its], 1), qp_iters=np.stack([a[1] for a in its], 1),
        step_status=np.stack([a[2] for a in its], 1)))


def assert_same_as_fused(mpc, x0, P, N, profile, mode, xb, k_sim, i_sim, **kw):
    ref = mpc.closed_loop(x0, P, N=N, k_sim=k_sim, i_sim=i_sim, profile=profile, want_Uk=True, state_rows=mode, xbounds=xb)
    got = controller_run_sc(mpc, x0, P, N, mode, xb, k_sim=k_sim, i_sim=i_sim, profile=profile, **kw)
    for key in ("xk", "uk", "Uk", "inner_iters", "qp_iters"):
        assert np.array_equal(got[key], ref[key], equal_nan=True), key
    st = got["step_status"].max(axis=1)
    st = np.where(np.isfinite(got["xk"]).all(axis=(1, 2)), st, np.maximum(st, 2))
    assert np.array_equal(st, ref["status"])
    return got, ref


# ------------------------------------------------------------------ 1. bit identity with the fused state-row loop
def _cases():
    base = [(3, 256, 0), (10, 256, 0), (20, 512, 0), (32, 256, 0),        # one warp, literal Gamma (Toeplitz rows)
            (40, 48, 0), (64, 32, 0), (72, 24, 0), (100, 16, 0),          # 2 and 4 warps, literal Gamma
            (10, 256, GAMMA_I), (20, 256, CONS), (32, 128, GAMMA_I),       # one warp, dense Gamma (DenseRows)
            (20, 256, DENSE_G), (10, 256, CONS), (32, 128, DENSE_G)]
    c, i = [], 0
    for N, S, prof in base:
        for mode in (REFRESH, FROZEN):
            fixed = i % 3 != 2                                          # every third case: the eps_break stop rule
            layout, host = (i // 2) % 2, i % 5 == 4
            xb = SCRIPT_BOX if N <= 32 and (i // 2) % 3 == 2 else XB
            name = (f"N{N}_{ {0: 'literal', GAMMA_I: 'gamma_i', CONS: 'consistent', DENSE_G: 'dense_g'}[prof]}"
                    f"_{'refresh' if mode == REFRESH else 'frozen'}_{'fixed' if fixed else 'eps'}_layout{layout}"
                    f"{'_host' if host else ''}_{'xb' if xb is XB else 'scriptbox'}")
            c.append((name, N, S, prof | (FIXED if fixed else 0), mode, xb, layout, host))
            i += 1
    return c


@pytest.mark.parametrize("name,N,S,profile,mode,xb,layout,host", _cases(), ids=[c[0] for c in _cases()])
def test_state_row_controller_steps_reproduce_the_fused_loop_bit_for_bit(mpc, name, N, S, profile, mode, xb, layout, host):
    P, x0, _ = batch(S, N)
    k_sim = 8 if N <= 32 else 4
    i_sim = 3 if profile & FIXED else 10
    got, ref = assert_same_as_fused(mpc, x0, P, N, profile, mode, xb, k_sim, i_sim, layout=layout, host=host)
    # the sample exercises the new ground: a scenario that ends infeasible, and one the rows steer off the box loop
    box = mpc.closed_loop(x0, P, N=N, k_sim=k_sim, i_sim=i_sim, profile=profile)
    assert (ref["status"] == INFEASIBLE).any()
    live = ~np.isnan(ref["uk"])
    assert (live & (ref["uk"] != box["uk"])).any()


# ------------------------------------------------------------------ 2. the infeasible step
@pytest.mark.parametrize("mode", [REFRESH, FROZEN])
def test_infeasible_step_returns_nan_and_leaves_the_record_alone(mpc, mode):
    import ntm_mpc
    P, x0, N = batch(256, 10)
    S = x0.shape[0]
    state = np.zeros((S, ntm_mpc.ctrl_doubles(N)))
    x, ended = x0.copy(), np.zeros(S, dtype=bool)
    seen_first = seen_later = 0
    for k in range(8):
        before = state.copy()
        r = mpc.mpc_step(state, x, P, N, 3, 1e-14, FIXED, want_U=True, state_rows=mode, xbounds=XB)
        bad = r["status"] == INFEASIBLE
        assert np.all(np.isnan(r["u"][bad])) and np.all(np.isnan(r["U"][bad]))
        assert np.all(np.isfinite(r["u"][~bad]))
        assert np.array_equal(state[bad].view(np.int64), before[bad].view(np.int64))      # bytes unchanged
        assert np.all(state[~bad, -1] == before[~bad, -1] + 1)                            # the others ran a step
        new = bad & ~ended
        seen_first += int(np.sum(new & (before[:, -1] == 0))); seen_later += int(np.sum(new & (before[:, -1] > 0)))
        ended |= bad
        xn = mpc.plant_step(x, r["u"], P)
        xn[ended] = x[ended]
        x = xn
    assert seen_first >= 1 and seen_later >= 1, (seen_first, seen_later)


# ------------------------------------------------------------------ 3. STATE_ROWS_OFF is ntm_mpc_step
@pytest.mark.parametrize("profile", [FIXED, GAMMA_I])
def test_state_rows_off_is_ntm_mpc_step_bit_for_bit(mpc, profile):
    import ntm_mpc
    P, x0, N = batch(512, 20)
    S = x0.shape[0]
    lib = mpc._lib
    sa, sb = np.zeros((S, ntm_mpc.ctrl_doubles(N))), np.zeros((S, ntm_mpc.ctrl_doubles(N)))
    x = x0.copy()
    for _ in range(10):
        outs = []
        for fn, st in (("a", sa), ("b", sb)):
            u, U = np.empty(S), np.empty((S, N))
            it = np.empty((3, S), dtype=np.int32)
            before = mpc.launch_count()
            args = (mpc._h, 0, profile, S, N, 10, 1e-14, x.ctypes.data, P.ctypes.data, S)
            tail = (st.ctypes.data, u.ctypes.data, U.ctypes.data, it[0].ctypes.data, it[1].ctypes.data, it[2].ctypes.data)
            rc = lib.ntm_mpc_step(*args, *tail) if fn == "a" else lib.ntm_mpc_step_sc(*args, 0, None, *tail)
            assert rc == 0 and mpc.launch_count() == before + 1
            outs.append((u, U, it))
        for a, b in zip(outs[0], outs[1]):
            assert np.array_equal(a, b)
        assert np.array_equal(sa.view(np.int64), sb.view(np.int64))
        x = mpc.plant_step(x, outs[0][0], P)


# ------------------------------------------------------------------ 4. restart
@pytest.mark.parametrize("mode,profile", [(FROZEN, FIXED), (REFRESH, FIXED), (FROZEN, GAMMA_I | FIXED)])
def test_zeroed_records_restart_from_a_new_x0_and_leave_the_others_alone(mpc, mode, profile):
    import ntm_mpc
    P, x0, N = batch(256, 10)
    S = x0.shape[0]
    xr = x0[::-1].copy()                                             # the restarted scenarios start somewhere else
    odd = np.arange(S) % 2 == 1
    K, R = 10, 4

    def run(xstart, restart_at=None):
        state, x, out = np.zeros((S, ntm_mpc.ctrl_doubles(N))), xstart.copy(), []
        for k in range(K):
            if k == restart_at:
                state[odd] = 0.0
                x[odd] = xr[odd]
            r = mpc.mpc_step(state, x, P, N, 3, 1e-14, profile, want_U=True, state_rows=mode, xbounds=XB)
            out.append(r)
            xn = mpc.plant_step(x, r["u"], P)
            dead = r["status"] == INFEASIBLE
            xn[dead] = x[dead]
            x = xn
        return out

    base, fresh, rs = run(x0), run(xr), run(x0, R)
    for k in range(K):
        for key in ("u", "U", "inner_iters", "qp_iters", "status"):
            assert np.array_equal(rs[k][key][~odd], base[k][key][~odd], equal_nan=key in ("u", "U")), (k, key)
            if k >= R:
                assert np.array_equal(rs[k][key][odd], fresh[k - R][key][odd], equal_nan=key in ("u", "U")), (k, key)
    # the restart matters: the odd scenarios' new trajectories differ from their old ones
    assert not np.array_equal(rs[R]["u"][odd], base[R]["u"][odd], equal_nan=True)


# ------------------------------------------------------------------ 5. a plant the fused loop cannot express
@pytest.mark.parametrize("N,mode", [(10, REFRESH), (10, FROZEN), (20, REFRESH), (20, FROZEN)])
def test_disturbed_plant_with_measurement_noise_and_state_rows_matches_the_oracle(mpc, N, mode):
    import ntm_mpc
    S, k_sim, i_sim = 32, 12, 3
    phys, x0, _ = o.make_batch(3, S=S)
    P = o.derive_params_batch(phys).T.copy()
    rng = np.random.default_rng(2000 + N + mode)
    dist = rng.normal(size=(k_sim, S, 2)) * np.array([5e-4, 30.0])           # additive plant disturbance on w, omega
    noise = rng.normal(size=(k_sim, S, 2)) * np.array([2e-4, 10.0])          # measurement noise seen by the controller
    state = np.zeros((S, ntm_mpc.ctrl_doubles(N)))
    x, gu, gst, ended = x0.copy(), [], [], np.zeros(S, dtype=bool)
    gx = [x0.copy()]
    for k in range(k_sim):
        r = mpc.mpc_step(state, x + noise[k], P, N, i_sim, profile=FIXED, state_rows=mode, xbounds=XB)
        ended |= r["status"] == INFEASIBLE
        u = np.where(ended, np.nan, r["u"])
        xn = mpc.plant_step(x, np.nan_to_num(u), P) + dist[k]
        x = np.where(ended[:, None], x, xn)
        gu.append(u); gx.append(np.where(ended[:, None], np.nan, x))
    gu, gx = np.stack(gu, 1), np.stack(gx, 1)
    prof = o.LITERAL_FIXED
    bad = n_inf = 0
    for s in range(S):
        p = o.scenario(phys, s)
        st, xo, ou, ox = {}, x0[s].copy(), [], [x0[s].copy()]
        for k in range(k_sim):
            r = controller_step_sc(p, st, xo + noise[k, s], N, i_sim, profile=prof, state_rows=mode, xbounds=XB)
            if r["status"] == INFEASIBLE:
                ou += [np.nan] * (k_sim - k); ox += [np.full(2, np.nan)] * (k_sim - k)
                break
            ou.append(r["u"])
            xo = o.plant_step(p, xo, ou[-1], prof) + dist[k, s]
            ox.append(xo)
        ou, ox = np.array(ou), np.array(ox)
        n_inf += int(np.isnan(ou).any())
        if not np.array_equal(np.isnan(gu[s]), np.isnan(ou)):                 # infeasible at another step
            bad += 1
            continue
        live = ~np.isnan(ou)
        if live.any():
            du = np.max(np.abs(gu[s][live] - ou[live])) / phys["umax"][s]
            w = ox[~np.isnan(ox[:, 0]), 0]
            dw = np.nanmax(np.abs(gx[s, :, 0] - ox[:, 0])) / max(np.max(np.abs(w)), 1e-3)
            bad += int(du > 1e-6 or dw > 1e-6)
    assert n_inf >= 1
    assert bad <= (1 if N > 20 else 0), bad


# ------------------------------------------------------------------ 6. contract
def test_one_launch_per_step_and_argument_checks(mpc):
    import ntm_mpc
    P, x0, N = batch(64, 20)
    S = x0.shape[0]
    for mode in (REFRESH, FROZEN):
        for prof in (0, GAMMA_I):
            state = np.zeros((S, ntm_mpc.ctrl_doubles(N)))
            for _ in range(3):
                before = mpc.launch_count()
                mpc.mpc_step(state, x0, P, N, state_rows=mode, xbounds=XB)
                assert mpc.launch_count() == before + 1
    lib = mpc._lib
    state = np.zeros((S, ntm_mpc.ctrl_doubles(128)))
    xp, pp, sp = x0.ctypes.data, P.ctypes.data, state.ctypes.data
    u = np.empty(S)
    xb = np.array(XB)

    def call(dev, profile=0, n=N, mode=REFRESH, b=xb):
        fn = lib.ntm_mpc_step_sc_dev if dev else lib.ntm_mpc_step_sc
        return fn(mpc._h, 0, profile, S, n, 10, 1e-14, xp, pp, S, mode, None if b is None else b.ctypes.data, sp,
                  u.ctypes.data, None, None, None, None)

    bad = [dict(profile=ntm_mpc.PROFILE_TAUE_W), dict(mode=3), dict(mode=-1), dict(b=None),
           dict(b=np.array([0.16, 0.05, 2000.0, 12000.0])), dict(b=np.array([0.05, 0.16, 12000.0, 2000.0])),
           dict(b=np.array([np.nan, 0.16, 2000.0, 12000.0])), dict(profile=GAMMA_I, n=40), dict(profile=DENSE_G, n=33),
           dict(n=128)]
    for dev in (False, True):
        for kw in bad:
            before = mpc.launch_count()
            assert call(dev, **kw) == 1, (dev, kw)
            assert lib.ntm_last_error().decode(), kw
            assert mpc.launch_count() == before, kw
    assert lib.ntm_mpc_step_sc_dev(mpc._h, 0, 0, 0, N, 10, 1e-14, None, None, 1, REFRESH, xb.ctypes.data, None, None,
                                   None, None, None, None) == 0


def test_caller_stream_without_host_sync_gives_the_same_bits(mpc):
    import torch
    P, x0, N = batch(512, 20)
    for mode in (REFRESH, FROZEN):
        ref = controller_run_sc(mpc, x0, P, N, mode, XB, profile=FIXED)
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            got = controller_run_sc(mpc, x0, P, N, mode, XB, profile=FIXED, stream=s)
        for key in ("xk", "uk", "Uk", "inner_iters", "qp_iters", "step_status"):
            assert np.array_equal(got[key], ref[key], equal_nan=True), key


def test_rows_warm_0_selects_the_cold_reference_for_controller_steps_too():
    """NTM_ROWS_WARM=0 (read once per process) starts every state-row QP cold, in the fused loop and in the step."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import sys, numpy as np\n"
        "sys.path[:0] = [%r, %r, %r]\n"
        "import ntm_mpc, test_gpu_controller_sc as t\n"
        "m = ntm_mpc.NtmMpc(0)\n"
        "P, x0, N = t.batch(256, 20)\n"
        "for mode in (1, 2):\n"
        "    t.assert_same_as_fused(m, x0, P, N, 16, mode, t.XB, 8, 3)\n"
        "print('cold identical')\n") % (os.path.join(root, "tests"), root, os.path.join(root, "mpc-ntm-control_b200"))
    env = dict(os.environ, NTM_ROWS_WARM="0")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=root)
    assert r.returncode == 0 and "cold identical" in r.stdout, r.stdout + r.stderr


# ------------------------------------------------------------------ 7. MEX gateway 11 against gateway 8
@pytest.mark.parametrize("mode", [REFRESH, FROZEN])
def test_mex_step_gateway_with_state_rows_and_host_plant_equals_ntm_mpc_batch(mpc, mode):
    from test_mex_gateway import Mock
    m = Mock()
    m.workspace({})
    P, x0, N = batch(256, 10)
    S, k_sim = x0.shape[0], 8
    lo, hi = np.array([XB[0], XB[2]]), np.array([XB[1], XB[3]])
    xk, uk, cost, inner, status = m.call("ntm_mpc_batch", [x0.T, P.T, N, k_sim, 10, 1e-14, FIXED, mode, lo, hi], nlhs=5)
    state, x = np.zeros((0, 0)), x0.copy()
    us, xs, sts, ended = [], [x0.copy()], [], np.zeros(S, dtype=bool)
    for _ in range(k_sim):
        u, state, U, inn, st = m.call("ntm_mpc_step", [state, x.T, P.T, N, 10, 1e-14, FIXED, mode, lo, hi], nlhs=5)
        ended |= st[0] == INFEASIBLE
        u = np.where(ended, np.nan, u[0])
        xn = mpc.plant_step(x, np.nan_to_num(u), P)
        x = np.where(ended[:, None], x, xn)
        us.append(u); xs.append(np.where(ended[:, None], np.nan, x)); sts.append(st[0])
    assert ended.any()
    assert np.array_equal(np.stack(us), uk, equal_nan=True)
    assert np.array_equal(np.stack(xs, 1).reshape(S, -1).T, xk, equal_nan=True)
    assert np.array_equal(np.where(ended, INFEASIBLE, np.max(sts, axis=0)), status[0])
