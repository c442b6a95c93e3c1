"""The receding-horizon controller step (ntm_mpc_step[_dev]) on the GPU (-m gpu).

k_sim controller steps, each followed by ntm_plant_step under the same profile, must reproduce the fused closed loop
(ntm_mpc_closed_loop) bit for bit on every instantiation the box-QP loop selects: one warp with the literal and the dense
Gamma (N <= 32, including the two-phase fused launch at 16,384 scenarios), the multi-warp dense row sweep, and the long
literal sweep tableau in registers and in shared memory.  Then a plant the fused loop cannot express (disturbances and
measurement noise) against the NumPy restatement, restarts of single scenarios, the C ABI contract, and MEX gateway 11."""

import numpy as np
import pytest

from controller_oracle import controller_step
from oracle import ntm_oracle as o

pytestmark = pytest.mark.gpu

FIXED, CONS = 16, 2 | 4 | 8


@pytest.fixture(scope="module")
def mpc():
    import ntm_mpc
    h = ntm_mpc.NtmMpc(0)
    yield h
    h.close()


def batch(cfg, S=None, N=None):
    phys, x0, n = o.make_batch(cfg, S=S)
    return o.derive_params_batch(phys).T.copy(), x0, (n if N is None else N)


def controller_run(mpc, x0, P, N, k_sim=20, i_sim=10, eps=1e-14, profile=0, layout=0, host=False, stream=None):
    """k_sim x (ntm_mpc_step[_dev] + ntm_plant_step[_dev]) on resident buffers; returns the fused loop's outputs."""
    import torch
    import ntm_mpc
    S = x0.shape[0]
    if host:
        state = np.zeros((S, ntm_mpc.ctrl_doubles(N)))
        x, out = x0.copy(), []
        for _ in range(k_sim):
            r = mpc.mpc_step(state, x, P, N, i_sim, eps, profile, want_U=True)
            out.append((x, r["u"], r["U"], r["inner_iters"], r["qp_iters"], r["status"]))
            x = mpc.plant_step(x, r["u"], P, profile)
        xs = [t[0] for t in out] + [x]
        return dict(xk=np.stack(xs, 1), uk=np.stack([t[1] for t in out], 1), Uk=np.stack([t[2] for t in out], 1),
                    inner_iters=np.stack([t[3] for t in out], 1), qp_iters=np.stack([t[4] for t in out], 1),
                    step_status=np.stack([t[5] for t in out], 1))
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
                         U.data_ptr(), it[0].data_ptr(), it[1].data_ptr(), it[2].data_ptr())
        xn = torch.empty_like(x)
        mpc.plant_step_dev(S, profile, layout, x.data_ptr(), u.data_ptr(), p.data_ptr(), S, xn.data_ptr())
        if stream is None:
            mpc.sync()
        hist.append((x, u.clone(), U.clone(), it.clone()))           # on the caller's stream: ordered, no host sync
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
    return dict(xk=np.stack(xs, 1), uk=np.stack([cpu(h[1]) for h in hist], 1), Uk=np.stack(Us, 1),
                inner_iters=np.stack([a[0] for a in its], 1), qp_iters=np.stack([a[1] for a in its], 1),
                step_status=np.stack([a[2] for a in its], 1))


def assert_same_as_fused(mpc, x0, P, N, profile, k_sim=20, **kw):
    ref = mpc.closed_loop(x0, P, N=N, k_sim=k_sim, profile=profile, want_Uk=True)
    got = controller_run(mpc, x0, P, N, k_sim=k_sim, profile=profile, **kw)
    for key in ("xk", "uk", "Uk", "inner_iters", "qp_iters"):
        assert np.array_equal(got[key], ref[key], equal_nan=True), key
    st = got["step_status"].max(axis=1)
    st = np.where(np.isfinite(got["xk"]).all(axis=(1, 2)), st, np.maximum(st, 2))
    assert np.array_equal(st, ref["status"])
    e = got["xk"][:, 1:, :] - P[:, None, 10:12]
    cost = np.sum(e[..., 0] * (P[:, None, 12] * e[..., 0] + P[:, None, 13] * e[..., 1])
                  + e[..., 1] * (P[:, None, 13] * e[..., 0] + P[:, None, 14] * e[..., 1]), axis=1)
    ok = np.isfinite(ref["cost"])
    assert np.all(np.abs(cost[ok] - ref["cost"][ok]) <= 1e-13 * np.abs(ref["cost"][ok])), "cost"
    return got


# ------------------------------------------------------------------ 4. bit identity with the fused loop
def _cases():
    c = [("config1_fixed", 1, None, None, FIXED, 0, False),
         ("config2_fixed_host", 2, None, None, FIXED, 0, True)]
    for prof in (FIXED, 0):
        for layout in (0, 1):
            c.append((f"config2_p{prof}_layout{layout}", 2, None, None, prof, layout, False))
    for prof in (FIXED, 0, CONS, 1):                           # 16,384 scenarios: the fused reference runs two-phase
        c.append((f"config3_16k_p{prof}", 3, 16384, None, prof, 0, False))
    c.append(("config4_4k", 4, 4096, None, FIXED, 0, False))
    c += [("N32_literal", 3, 512, 32, 0, 0, False), ("N32_gamma_i", 3, 512, 32, 2, 0, False),
          ("N48_gamma_i", 3, 256, 48, 2, 0, False), ("N80_gamma_i", 3, 64, 80, 2, 0, False),
          ("N64_gamma_i_row_sweep", 3, 64, 64, 2, 0, False), ("N120_gamma_i_row_sweep", 3, 32, 120, 2, 0, False)]
    for N in (40, 64, 100, 110):                              # long literal paths: tableau in registers / shared memory
        c.append((f"config5_N{N}", 5, 512, N, FIXED, 0, False))
    return c


@pytest.mark.parametrize("name,cfg,S,N,profile,layout,host", _cases(), ids=[c[0] for c in _cases()])
def test_controller_steps_reproduce_the_fused_loop_bit_for_bit(mpc, name, cfg, S, N, profile, layout, host):
    P, x0, n = batch(cfg, S, N)
    assert_same_as_fused(mpc, x0, P, n, profile, layout=layout, host=host)


def test_plant_only_profile_bits_have_no_effect_on_the_controller(mpc):
    P, x0, N = batch(2, 256)
    a = controller_run(mpc, x0, P, N, k_sim=1, profile=0)
    for extra in (8, 64, 8 | 64):
        b = controller_run(mpc, x0, P, N, k_sim=1, profile=extra)
        assert np.array_equal(a["uk"], b["uk"]) and np.array_equal(a["Uk"], b["Uk"])


# ------------------------------------------------------------------ 5. a plant the fused loop cannot express
@pytest.mark.parametrize("N,S", [(3, 64), (10, 64), (20, 64), (40, 16)])
def test_disturbed_plant_with_measurement_noise_matches_the_oracle(mpc, N, S):
    import ntm_mpc
    phys, x0, _ = o.make_batch(3, S=S)
    P = o.derive_params_batch(phys).T.copy()
    rng = np.random.default_rng(1000 + N)
    k_sim = 20
    dist = rng.normal(size=(k_sim, S, 2)) * np.array([5e-4, 30.0])           # additive plant disturbance on w, omega
    noise = rng.normal(size=(k_sim, S, 2)) * np.array([2e-4, 10.0])          # measurement noise seen by the controller
    state = np.zeros((S, ntm_mpc.ctrl_doubles(N)))
    x, gu, gx = x0.copy(), [], [x0.copy()]
    for k in range(k_sim):
        u = mpc.mpc_step(state, x + noise[k], P, N, profile=FIXED)["u"]
        x = mpc.plant_step(x, u, P) + dist[k]
        gu.append(u); gx.append(x)
    gu, gx = np.stack(gu, 1), np.stack(gx, 1)
    prof = o.LITERAL_FIXED
    bad = 0
    for s in range(S):
        p = o.scenario(phys, s)
        st, xo, ou, ox = {}, x0[s].copy(), [], [x0[s].copy()]
        for k in range(k_sim):
            ou.append(controller_step(p, st, xo + noise[k, s], N, profile=prof)["u"])
            xo = o.plant_step(p, xo, ou[-1], prof) + dist[k, s]
            ox.append(xo)
        ou, ox = np.array(ou), np.array(ox)
        du = np.max(np.abs(gu[s] - ou)) / phys["umax"][s]
        dw = np.max(np.abs(gx[s, :, 0] - ox[:, 0])) / max(np.max(np.abs(ox[:, 0])), 1e-3)
        bad += int(du > 1e-6 or dw > 1e-6)
    assert bad <= (1 if N > 20 else 0), bad


# ------------------------------------------------------------------ 6. restart and independence
def test_zeroed_records_restart_their_scenarios_and_leave_the_others_alone(mpc):
    import ntm_mpc
    P, x0, N = batch(2, 256)
    S = x0.shape[0]
    odd = np.arange(S) % 2 == 1

    def run(restart_at):
        state, x, out = np.zeros((S, ntm_mpc.ctrl_doubles(N))), x0.copy(), []
        for k in range(20):
            if k == restart_at:
                state[odd] = 0.0
                x[odd] = x0[odd]
            r = mpc.mpc_step(state, x, P, N, profile=FIXED, want_U=True)
            out.append(r)
            x = mpc.plant_step(x, r["u"], P)
        return out

    base, rs = run(None), run(10)
    for k in range(20):
        for key in ("u", "U", "inner_iters", "qp_iters", "status"):
            assert np.array_equal(rs[k][key][~odd], base[k][key][~odd]), (k, key)
            if k >= 10:
                assert np.array_equal(rs[k][key][odd], base[k - 10][key][odd]), (k, key)


# ------------------------------------------------------------------ 7. contract
def test_one_launch_per_step_and_argument_checks(mpc):
    import ntm_mpc
    P, x0, N = batch(2, 64)
    S = x0.shape[0]
    state = np.zeros((S, ntm_mpc.ctrl_doubles(N)))
    for _ in range(3):
        before = mpc.launch_count()
        mpc.mpc_step(state, x0, P, N)
        assert mpc.launch_count() == before + 1
    lib = mpc._lib
    xp, pp, sp = x0.ctypes.data, P.ctypes.data, state.ctypes.data
    u = np.empty(S)

    def call(profile=0, n=N, s=S, st=sp, i_sim=10):
        return lib.ntm_mpc_step(mpc._h, 0, profile, s, n, i_sim, 1e-14, xp, pp, s, st, u.ctypes.data, None, None, None, None)

    for kw in (dict(profile=ntm_mpc.PROFILE_TAUE_W), dict(n=0), dict(n=129), dict(st=None), dict(i_sim=0)):
        assert call(**kw) == 1, kw
        assert lib.ntm_last_error().decode(), kw
    before = mpc.launch_count()
    assert call(s=0, st=None) == 0 and mpc.launch_count() == before
    assert lib.ntm_mpc_step_dev(mpc._h, 0, 0, 0, N, 10, 1e-14, None, None, 1, None, None, None, None, None, None) == 0


def test_caller_stream_without_host_sync_gives_the_same_bits(mpc):
    import torch
    P, x0, N = batch(2)
    ref = controller_run(mpc, x0, P, N, profile=FIXED)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got = controller_run(mpc, x0, P, N, profile=FIXED, stream=s)
    for key in ("xk", "uk", "Uk", "inner_iters", "qp_iters", "step_status"):
        assert np.array_equal(got[key], ref[key]), key


# ------------------------------------------------------------------ 8. MEX gateway 11
def test_mex_step_gateway_with_host_plant_equals_ntm_mpc_batch(mpc):
    from test_mex_gateway import Mock
    m = Mock()
    m.workspace({})
    P, x0, N = batch(2)
    S, k_sim = x0.shape[0], 20
    xk, uk = m.call("ntm_mpc_batch", [x0.T, P.T, N, k_sim, 10, 1e-14, FIXED], nlhs=2)
    state, x, us, xs = np.zeros((0, 0)), x0.copy(), [], [x0.copy()]
    for _ in range(k_sim):
        u, state, U, inner, status = m.call("ntm_mpc_step", [state, x.T, P.T, N, 10, 1e-14, FIXED], nlhs=5)
        assert state.shape == (7 * N + 7, S) and U.shape == (N, S) and np.all(inner == 10)
        x = mpc.plant_step(x, u[0], P)
        us.append(u[0]); xs.append(x)
    assert np.array_equal(np.stack(us), uk)
    assert np.array_equal(np.concatenate(xs, axis=1).T, xk)
