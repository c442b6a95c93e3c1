"""The state observer on the GPU (-m gpu): ntm_kf_step[_dev] and ntm_mpc_closed_loop_observed[_dev].

1. ntm_kf_step against the NumPy twin (tests/observer_oracle.py) to 1e-12 relative on xhat and P: both layouts, host and
   device entries, one or S parameter blocks, batch sizes that wrap the grid, fresh, resumed and partially zeroed records.
2. The observed loop is bit-identical to the step-API composition k_sim x (ntm_kf_step at y_k = x_k + v_k,
   ntm_mpc_step_sc at xhat_k, ntm_plant_step + d_k), up to and including each scenario's infeasible step, on every
   instantiation the perturbed loop has (one warp literal / dense Gamma, multi-warp dense, long tableau in registers and
   in shared memory, state rows off, refreshed and frozen on every row instantiation).
3. Nothing perturbed: bit-identical to ntm_mpc_closed_loop / ntm_mpc_closed_loop_sc, with xhat = xk(:, 0..k_sim-1).
4. The filter filters (see test_the_estimate_is_closer_to_the_state_than_the_measurement).
5. Scenarios stay independent, one launch per call, argument errors launch nothing, the caller's stream.
6. montecarlo.run(kf_cov=...) and MEX gateways 12 and 13 against the C ABI."""

import numpy as np
import pytest

from oracle import ntm_oracle as o
from observer_oracle import kf_step as twin_kf_step
from test_gpu_perturbed import blocks, host_cost, same_bits

pytestmark = pytest.mark.gpu

RHO1_SQ, GAMMA_I, F_XK, PLANT_C, FIXED, DENSE_G, RK4, TAUE_W = 1, 2, 4, 8, 16, 32, 64, 128
OFF, REFRESH, FROZEN = 0, 1, 2
KEYS = ("xk", "uk", "Uk", "xhat", "inner_iters", "qp_iters", "status")
XB = (0.05, 0.16, 2000.0, 12000.0)          # binds on part of config 3 and is infeasible on another
KC = np.array([1e-6, 0.0, 900.0, 2.5e-7, 0.0, 400.0])   # kf_cov_from_std((1e-3, 30), (5e-4, 20))


@pytest.fixture(scope="module")
def mpc():
    import ntm_mpc
    h = ntm_mpc.NtmMpc(0)
    yield h
    h.close()


def noise(S, k_sim, seed=5):
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(S, k_sim, 2)) * np.array([4e-3, 600.0])     # large enough that true states leave the box and
    v = rng.normal(size=(S, k_sim, 2)) * np.array([5e-3, 500.0])     # that estimates alone end some scenarios
    return d, v


def to_profile(flags):
    return o.Profile(rho1_variant=flags & 1, gamma_index=(flags >> 1) & 1, f_state=(flags >> 2) & 1,
                     plant_affine=(flags >> 3) & 1, inner_policy=(flags >> 4) & 1, plant_integrator=(flags >> 6) & 1)


# ---------------------------------------------------------------------------------------------------------- kf step
def kf_dev(mpc, state, y, u, P, kc, profile, layout):
    """ntm_kf_step_dev on resident buffers: y in `layout`, records scenario slowest; updates `state` like the host
    entry and returns xhat [S, 2]."""
    import torch
    import ntm_mpc
    dev = torch.device("cuda")
    soa = layout == ntm_mpc.LAYOUT_SOA
    S = y.shape[0]
    put = lambda a: torch.tensor(np.ascontiguousarray(a.T if soa else a), device=dev)
    dy, du, dP = put(y), torch.tensor(u, device=dev), put(np.atleast_2d(P))
    dst = torch.tensor(state, device=dev)
    dx = torch.empty(2 * S, dtype=torch.float64, device=dev)
    mpc.kf_step_dev(S, profile, layout, dy.data_ptr(), du.data_ptr(), dP.data_ptr(), P.shape[0] if P.ndim == 2 else 1,
                    kc, dst.data_ptr(), dx.data_ptr())
    mpc.sync()
    state[:] = dst.cpu().numpy()
    x = dx.cpu().numpy()
    return x.reshape(2, S).T.copy() if soa else x.reshape(S, 2)


def close_records(got, ref, rtol=1e-12):
    """xhat to rtol relative; P to rtol of sqrt(p_ii p_jj); steps exactly."""
    ok = np.all(np.abs(got[:, :2] - ref[:, :2]) <= rtol * np.abs(ref[:, :2]))
    s11, s22 = np.abs(ref[:, 2]), np.abs(ref[:, 4])
    scale = np.stack([s11, np.sqrt(s11 * s22), s22], axis=1)
    ok &= np.all(np.abs(got[:, 2:5] - ref[:, 2:5]) <= rtol * scale)
    return bool(ok and np.array_equal(got[:, 5], ref[:, 5]))


KF_CASES = [(S, layout, entry, pcs, prof) for S, layout, entry, pcs, prof in [
    (1, 0, "host", False, 0), (255, 1, "dev", True, RK4 | PLANT_C), (257, 0, "dev", False, RHO1_SQ),
    (257, 1, "host", True, FIXED | GAMMA_I), (65537, 0, "dev", True, RK4), (65537, 1, "host", False, PLANT_C)]]


@pytest.mark.parametrize("S,layout,entry,pcs,prof", KF_CASES,
                         ids=[f"S{c[0]}-L{c[1]}-{c[2]}-pc{'S' if c[3] else '1'}-p{c[4]}" for c in KF_CASES])
def test_kf_step_matches_the_twin(mpc, S, layout, entry, pcs, prof):
    base = min(S, 4096)
    phys, x0, _ = o.make_batch(3, S=base, seed=21)
    idx = np.arange(S) % base
    P = o.derive_params_batch(phys).T[idx].copy()
    x = x0[idx]
    if not pcs:
        P = P[0].copy()
    rng = np.random.default_rng(S)
    profile = to_profile(prof)
    check = np.unique(np.concatenate([np.arange(min(S, 300)), np.arange(max(S - 300, 0), S),
                                      rng.choice(S, min(S, 1500), replace=False)]))
    state = np.zeros((S, 6))
    ref = np.zeros((S, 6))
    u = rng.uniform(0.0, 2e6, size=S)
    for step in range(4):
        if step == 2:                                    # partially zeroed: those records start again
            z = rng.random(S) < 0.3
            z[0] = True
            state[z] = 0.0; ref[z] = 0.0
        y = x + rng.normal(size=(S, 2)) * np.array([5e-4, 20.0])
        if entry == "host":
            xh = mpc.kf_step(state, y, u, P, KC, prof)
        else:
            xh = kf_dev(mpc, state, y, u, P, KC, prof, layout)
        assert same_bits(xh, state[:, :2])
        for s in check:
            p = o.scenario(phys, int(idx[s]) if pcs else 0)      # one shared block: scenario 0's
            ref[s] = twin_kf_step(p, ref[s], y[s], u[s], KC, profile)
        assert close_records(state[check], ref[check]), step
        x = x + rng.normal(size=(S, 2)) * np.array([1e-3, 30.0])
        u = rng.uniform(0.0, 2e6, size=S)
    assert set(np.unique(state[:, 5])) <= {2.0, 4.0} and np.any(state[:, 5] == 2.0)
    P11, P21, P22 = state[:, 2], state[:, 3], state[:, 4]
    assert np.all(P11 > 0) and np.all(P22 > 0) and np.all(P11 * P22 - P21 ** 2 >= 0)


def test_kf_step_layouts_and_entries_give_the_same_bits(mpc):
    import ntm_mpc
    S = 300
    P, _, x0 = blocks(S)
    rng = np.random.default_rng(2)
    ys = [x0 + rng.normal(size=(S, 2)) * np.array([5e-4, 20.0]) for _ in range(3)]
    outs = []
    for layout, entry in ((0, "host"), (0, "dev"), (1, "dev")):
        state = np.zeros((S, 6))
        for k in range(3):
            y, u = ys[k], np.full(S, 1e5 * k)             # the input applied since the last step (ignored at k = 0)
            if entry == "host":
                mpc.kf_step(state, y, u, P, KC, RK4)
            else:
                kf_dev(mpc, state, y, u, P, KC, RK4, layout)
        outs.append(state.copy())
    assert same_bits(outs[0], outs[1]) and same_bits(outs[0], outs[2])
    # an observer drives the same records
    obs = mpc.observer(P, KC, profile=RK4)
    u = None
    for k in range(3):
        obs.update(ys[k], u)
        u = np.full(S, 1e5 * (k + 1))
    assert same_bits(obs.state, outs[0])
    assert ntm_mpc.kf_doubles() == obs.state.shape[1]


# ---------------------------------------------------------------------------------------------------------- the loop
def composition(mpc, x0, P, N, k_sim, i_sim, eps, profile, PP, pprof, d, v, mode, xb, kc=KC):
    """The contract, written out with the step API: ntm_kf_step at y_k = x_k + v_k and u_{k-1}, ntm_mpc_step_sc at
    xhat_k, ntm_plant_step, + d_k; a scenario whose step comes back infeasible ends there (NaN u, U, later states and
    estimates, iteration counts 0 after it).  Returns the final filter records too."""
    import ntm_mpc
    S = x0.shape[0]
    state = np.zeros((S, ntm_mpc.ctrl_doubles(N)))
    kfs = np.zeros((S, 6))
    x = x0.copy()
    xk = np.full((S, k_sim + 1, 2), np.nan); xk[:, 0] = x0
    xhat = np.full((S, k_sim, 2), np.nan)
    uk = np.full((S, k_sim), np.nan); Uk = np.full((S, k_sim, N), np.nan)
    inner = np.zeros((S, k_sim), dtype=np.int32); qpit = np.zeros((S, k_sim), dtype=np.int32)
    status = np.zeros(S, dtype=np.int32)
    live = np.ones(S, dtype=bool)
    k_inf = np.full(S, -1)
    u_prev = np.zeros(S)
    for k in range(k_sim):
        y = x if v is None else x + v[:, k]
        xh = mpc.kf_step(kfs, np.where(live[:, None], y, 0.1), u_prev, P, kc, profile)
        xhat[live, k] = xh[live]
        r = mpc.mpc_step(state, np.where(live[:, None], xh, 0.1), P, N, i_sim, eps, profile, want_U=True,
                         state_rows=mode, xbounds=xb)
        inner[live, k] = r["inner_iters"][live]; qpit[live, k] = r["qp_iters"][live]
        status[live] = np.maximum(status[live], r["status"][live])
        dead = live & (r["status"] == 3)
        k_inf[dead] = k
        live &= ~dead
        xn = mpc.plant_step(x, np.where(live, r["u"], 0.0), PP, pprof)
        if d is not None:
            xn = xn + d[:, k]
        x = np.where(live[:, None], xn, x)
        xk[live, k + 1] = x[live]; uk[live, k] = r["u"][live]; Uk[live, k] = r["U"][live]
        u_prev = np.where(live, r["u"], 0.0)
    fin = live & ~np.all(np.isfinite(xk[:, -1]), axis=1)
    status[fin] = np.maximum(status[fin], 2)
    return dict(xk=xk, uk=uk, Uk=Uk, xhat=xhat, inner_iters=inner, qp_iters=qpit, status=status, k_inf=k_inf, kf=kfs)


def observed_dev(mpc, x0, P, N, k_sim, i_sim, eps, profile, PP, pprof, d, v, layout, mode, xb, kc=KC, stream=None):
    """The _dev entry on resident buffers in `layout`; returns host arrays shaped like the host entry's."""
    import torch
    import ntm_mpc
    dev = torch.device("cuda")
    soa = layout == ntm_mpc.LAYOUT_SOA
    S = x0.shape[0]

    def put(a, E):                       # [S, E] (flattened per scenario) -> device array in `layout`
        if a is None:
            return None
        a = np.ascontiguousarray(a).reshape(-1, E)
        return torch.tensor(a.T.copy() if soa else a, device=dev)

    x = put(x0, 2); p = put(P, ntm_mpc.NPARAM); pp = put(PP, ntm_mpc.NPARAM) if PP is not None else None
    dw = put(d, 2 * k_sim); dv = put(v, 2 * k_sim)
    f64 = dict(dtype=torch.float64, device=dev)
    xk = torch.empty(S * 2 * (k_sim + 1), **f64); uk = torch.empty(S * k_sim, **f64)
    Uk = torch.empty(S * N * k_sim, **f64); cost = torch.empty(S, **f64); xh = torch.empty(S * 2 * k_sim, **f64)
    i32 = dict(dtype=torch.int32, device=dev)
    inner = torch.empty(S * k_sim, **i32); qp = torch.empty(S * k_sim, **i32); st = torch.empty(S, **i32)
    torch.cuda.synchronize()
    if stream is not None:
        mpc.set_stream(stream.cuda_stream)
    ptr = lambda t: 0 if t is None else t.data_ptr()
    count = lambda B: B.shape[0] if B.ndim == 2 else 1
    mpc.closed_loop_observed_dev(S, N, k_sim, i_sim, eps, profile, layout, ptr(x), ptr(p), count(P),
                                 ptr(pp), count(PP) if PP is not None else 0, pprof,
                                 ptr(dw), ptr(dv), ptr(xk), ptr(uk), ptr(Uk), ptr(cost), ptr(inner), ptr(qp), ptr(st),
                                 state_rows=mode, xbounds=xb, kf_cov=kc, xhat_ptr=ptr(xh))
    if stream is not None:
        stream.synchronize()
        mpc.reset_stream()
    mpc.sync()

    def get(t, E):
        a = t.cpu().numpy()
        return a.reshape(E, S).T.copy() if soa else a.reshape(S, E)
    return dict(xk=get(xk, 2 * (k_sim + 1)).reshape(S, k_sim + 1, 2), uk=get(uk, k_sim),
                Uk=get(Uk, N * k_sim).reshape(S, k_sim, N), xhat=get(xh, 2 * k_sim).reshape(S, k_sim, 2),
                cost=cost.cpu().numpy(), inner_iters=get(inner, k_sim), qp_iters=get(qp, k_sim), status=st.cpu().numpy())


# N, profile, plant_profile, per-scenario controller block, per-scenario plant block, layout, entry, rows, d / v
CASES = [
    (3, FIXED, 0, False, True, 0, "host", REFRESH, True),                    # one warp, literal Gamma, rows
    (10, RK4, RK4, True, True, 1, "dev", FROZEN, True),
    (20, FIXED | PLANT_C, TAUE_W, True, False, 0, "dev", REFRESH, True),
    (32, RHO1_SQ, PLANT_C | RHO1_SQ, True, True, 0, "host", FROZEN, True),
    (24, GAMMA_I | FIXED, RHO1_SQ, True, True, 0, "dev", REFRESH, True),     # one warp, dense Gamma, rows
    (16, GAMMA_I | RK4, RK4, False, True, 1, "dev", FROZEN, True),
    (30, DENSE_G, TAUE_W, True, True, 0, "host", FROZEN, True),
    (40, FIXED, RK4, True, True, 0, "dev", REFRESH, True),                   # two / four warps, literal Gamma, rows
    (64, 0, TAUE_W, True, True, 1, "dev", FROZEN, True),
    (100, FIXED | RK4 | PLANT_C, PLANT_C | RK4, True, True, 1, "dev", FROZEN, True),
    (100, 0, 0, True, False, 0, "host", REFRESH, True),
    (20, FIXED, RK4, True, True, 0, "host", OFF, True),                      # box QP: one warp literal / dense
    (12, GAMMA_I | PLANT_C, TAUE_W, True, True, 1, "dev", OFF, True),
    (40, GAMMA_I | FIXED, RK4, True, True, 1, "dev", OFF, True),             # multi-warp dense
    (90, DENSE_G, 0, True, False, 0, "host", OFF, True),
    (48, FIXED | RK4, TAUE_W, True, True, 0, "dev", OFF, True),              # long tableau in registers
    (100, RHO1_SQ, RHO1_SQ | PLANT_C, True, True, 1, "host", OFF, True),
    (120, FIXED, RK4, True, True, 1, "dev", OFF, True),                      # long tableau in shared memory
    (20, FIXED, 0, True, True, 0, "dev", OFF, False),
]


@pytest.mark.parametrize("N,profile,pprof,pc_s,ppc_s,layout,entry,mode,pert", CASES,
                         ids=[f"N{c[0]}-p{c[1]}-pp{c[2]}-{c[6]}-L{c[5]}-r{c[7]}-{'dv' if c[8] else 'nodv'}" for c in CASES])
def test_bit_identical_to_the_step_composition(mpc, N, profile, pprof, pc_s, ppc_s, layout, entry, mode, pert):
    S, k_sim, i_sim, eps = 64, 8, 4, 1e-14
    P, PP, x0 = blocks(S)
    if not pc_s:
        P = P[0]
    if not ppc_s:
        PP = PP[3]
    d, v = noise(S, k_sim) if pert else (None, None)
    ref = composition(mpc, x0, P, N, k_sim, i_sim, eps, profile, PP, pprof, d, v, mode, XB)
    if entry == "host":
        got = mpc.closed_loop_observed(x0, P, N, KC, plant_params=PP, plant_profile=pprof, w=d, v=v, k_sim=k_sim,
                                       i_sim=i_sim, eps=eps, profile=profile, want_Uk=True, state_rows=mode, xbounds=XB)
    else:
        got = observed_dev(mpc, x0, P, N, k_sim, i_sim, eps, profile, PP, pprof, d, v, layout, mode, XB)
    for key in KEYS:
        assert same_bits(got[key], ref[key]), key
    ended = ref["k_inf"] >= 0
    assert np.all(np.isnan(got["cost"][ended]))
    assert np.allclose(got["cost"][~ended], host_cost(got["xk"][~ended], np.broadcast_to(P, (S, P.shape[-1]))[~ended]),
                       rtol=1e-13, atol=0)
    if mode != OFF:
        assert np.any(ended)
        for s in np.nonzero(ended)[0]:
            assert np.all(np.isnan(got["xhat"][s, ref["k_inf"][s] + 1:]))
            assert np.all(np.isfinite(got["xhat"][s, :ref["k_inf"][s] + 1]))
    if pert:                                      # the controller did see something else than y_k
        y = got["xk"][:, :k_sim] + v
        fin = np.isfinite(got["xhat"][:, 1:])
        assert np.any(fin & (got["xhat"][:, 1:] != y[:, 1:]))


# nothing perturbed: the estimate is the state itself
UNPERTURBED = [(None, 20, 0, OFF, None), (None, 20, FIXED, REFRESH, None), (512, 20, 0, FROZEN, XB),
               (512, 10, RK4 | PLANT_C | RHO1_SQ, REFRESH, XB), (512, 24, GAMMA_I, FROZEN, XB),
               (512, 40, GAMMA_I | FIXED, OFF, None), (256, 48, RK4, OFF, None), (256, 100, FIXED, REFRESH, XB),
               (256, 120, PLANT_C, OFF, None)]


@pytest.mark.parametrize("S,N,profile,mode,xb", UNPERTURBED,
                         ids=[f"S{c[0]}-N{c[1]}-p{c[2]}-r{c[3]}" for c in UNPERTURBED])
def test_no_perturbation_is_the_closed_loop(mpc, S, N, profile, mode, xb):
    phys, x0, _ = o.make_batch(3, S=S)
    P = o.derive_params_batch(phys).T.copy()
    ref = mpc.closed_loop(x0, P, N, profile=profile, want_Uk=True, state_rows=mode, xbounds=xb)
    kc = np.array([3e-7, 1e-4, 400.0, 1e-6, -2e-3, 900.0])
    got = mpc.closed_loop_observed(x0, P, N, kc, profile=profile, want_Uk=True, state_rows=mode, xbounds=xb)
    for key in ("xk", "uk", "Uk", "inner_iters", "qp_iters", "status", "cost"):
        assert same_bits(got[key], ref[key]), key
    live = np.isfinite(got["xhat"])
    assert same_bits(got["xhat"][live], ref["xk"][:, :-1][live])
    assert np.array_equal(live, np.isfinite(ref["xk"][:, :-1]))


def test_the_estimate_is_closer_to_the_state_than_the_measurement(mpc):
    """Config 3 draws, 4,096 scenarios, N = 20, the nominal plant, measurement noise dominant over the process
    disturbance, kf_cov matched to both: over every step after the first, RMS(xhat - x) < RMS(y - x) per component.
    Measured on one NVIDIA B200: RMS(xhat - x) / RMS(y - x) = 0.4545 for w and 0.4142 for omega.  The step-API
    composition on the same draws gives the same bits and leaves every P symmetric with det P >= 0."""
    from ntm_mpc import montecarlo
    S, k_sim = 4096, 20
    phys, x0, N = o.make_batch(3, S=S)
    P = o.derive_params_batch(phys).T.copy()
    w_std, v_std = np.array([1e-4, 3.0]), np.array([5e-4, 20.0])
    rng = np.random.default_rng(17)
    d = rng.normal(size=(S, k_sim, 2)) * w_std
    v = rng.normal(size=(S, k_sim, 2)) * v_std
    kc = montecarlo.kf_cov_from_std(w_std, v_std)
    got = mpc.closed_loop_observed(x0, P, N, kc, w=d, v=v, k_sim=k_sim, profile=FIXED, want_Uk=True)
    x = got["xk"][:, 1:k_sim]
    e_hat = got["xhat"][:, 1:] - x
    e_y = v[:, 1:]
    ok = np.all(np.isfinite(e_hat), axis=(1, 2))
    assert ok.mean() > 0.99
    rms = lambda e: np.sqrt(np.mean(e[ok] ** 2, axis=(0, 1)))
    ratio = rms(e_hat) / rms(e_y)
    print(f"RMS(xhat - x) / RMS(y - x): w {ratio[0]:.4f}, omega {ratio[1]:.4f}")
    assert np.all(ratio < 1.0), ratio
    ref = composition(mpc, x0, P, N, k_sim, 10, 1e-14, FIXED, P, 0, d, v, OFF, None, kc)
    for key in KEYS:
        assert same_bits(got[key], ref[key]), key
    kf = ref["kf"]
    assert np.all(kf[:, 2] >= 0) and np.all(kf[:, 4] >= 0) and np.all(kf[:, 2] * kf[:, 4] - kf[:, 3] ** 2 >= 0)
    assert np.all(kf[:, 5] == k_sim)


def test_scenarios_stay_independent(mpc):
    S, N, k_sim = 32, 20, 8
    P, PP, x0 = blocks(S)
    d, v = noise(S, k_sim)
    kw = dict(plant_profile=RK4, k_sim=k_sim, state_rows=FROZEN, xbounds=XB, want_Uk=True)
    base = mpc.closed_loop_observed(x0, P, N, KC, plant_params=PP, w=d, v=v, **kw)
    v2 = v.copy()
    v2[9, 2, 1] = np.nan
    got = mpc.closed_loop_observed(x0, P, N, KC, plant_params=PP, w=d, v=v2, **kw)
    keep = np.setdiff1d(np.arange(S), [9])
    for key in KEYS + ("cost",):
        assert same_bits(got[key][keep], base[key][keep]), key
    assert got["status"][9] >= 2 and np.all(np.isnan(got["xhat"][9, 2:]))
    perm = np.random.default_rng(4).permutation(S)
    pg = mpc.closed_loop_observed(x0[perm], P[perm], N, KC, plant_params=PP[perm], w=d[perm], v=v[perm], **kw)
    for key in KEYS + ("cost",):
        assert same_bits(pg[key], base[key][perm]), key


def test_one_launch_argument_errors_and_the_callers_stream(mpc):
    import torch
    import ntm_mpc
    S, N, k_sim = 16, 12, 5
    P, PP, x0 = blocks(S)
    d, v = noise(S, k_sim)
    args = (mpc, x0, P, N, k_sim, 10, 1e-14, 0, PP, RK4, d, v, 0, REFRESH, XB)
    ref = observed_dev(*args)
    before = mpc.launch_count()
    observed_dev(*args)
    assert mpc.launch_count() == before + 1
    before = mpc.launch_count()
    host = mpc.closed_loop_observed(x0, P, N, KC, plant_params=PP, plant_profile=RK4, w=d, v=v, k_sim=k_sim,
                                    want_Uk=True, state_rows=REFRESH, xbounds=XB)
    assert mpc.launch_count() == before + 1
    for key in KEYS + ("cost",):
        assert same_bits(host[key], ref[key]), key
    state = np.zeros((S, 6))
    before = mpc.launch_count()
    mpc.kf_step(state, x0, np.zeros(S), P, KC)
    kf_dev(mpc, state, x0, np.zeros(S), P, KC, 0, 1)
    assert mpc.launch_count() == before + 2
    s = torch.cuda.Stream()
    got = observed_dev(*args, stream=s)
    for key in KEYS + ("cost",):
        assert same_bits(got[key], ref[key]), key
    # argument errors, through the C entries themselves (the Python front end refuses some of them first): nothing
    # launched, nothing copied (the host entry's output arrays stay as they were)
    lib = mpc._lib
    before = mpc.launch_count()
    bad_cov = [None, KC[:5].tolist() + [np.nan], [1e-6, 0.0, -1.0, 2.5e-7, 0.0, 400.0], [1e-6, 1.0, 900.0, 2.5e-7, 0.0, 400.0],
               [1e-6, 0.0, 900.0, 0.0, 0.0, 400.0], [1e-6, 0.0, 900.0, 2.5e-7, 1.0, 400.0], [1e-6, 0.0, 900.0, 2.5e-7, 0.0, -1.0]]
    bad = [dict(kc=c) for c in bad_cov] + [dict(profile=TAUE_W), dict(plant_profile=GAMMA_I), dict(state_rows=3),
                                          dict(xbounds=np.array([0.16, 0.05, 2000.0, 12000.0])), dict(N=129), dict(ppc=2)]
    for b in bad:
        a = dict(profile=0, plant_profile=RK4, state_rows=REFRESH, xbounds=np.array(XB), N=N, ppc=S, kc=KC)
        a.update(b)
        kc = None if a["kc"] is None else np.asarray(a["kc"], dtype=np.float64)
        kcp = None if kc is None else kc.ctypes.data
        xb = a["xbounds"].ctypes.data
        xk = np.full((S, k_sim + 1, 2), 7.0); uk = np.full((S, k_sim), 7.0); xh = np.full((S, k_sim, 2), 7.0)
        rc = lib.ntm_mpc_closed_loop_observed(mpc._h, ntm_mpc.LAYOUT_MATLAB, a["profile"], S, a["N"], k_sim, 10, 1e-14,
                                              x0.ctypes.data, P.ctypes.data, S, a["state_rows"], xb, PP.ctypes.data,
                                              a["ppc"], a["plant_profile"], d.ctypes.data, v.ctypes.data, kcp,
                                              xh.ctypes.data, xk.ctypes.data, uk.ctypes.data, None, None, None, None, None)
        assert rc != 0, b
        assert np.all(xk == 7.0) and np.all(uk == 7.0) and np.all(xh == 7.0), b
        rc = lib.ntm_mpc_closed_loop_observed_dev(mpc._h, 0, a["profile"], S, a["N"], k_sim, 10, 1e-14, 1, 1, 1,
                                                  a["state_rows"], xb, 1, a["ppc"], a["plant_profile"], None, None, kcp,
                                                  1, 1, 1, None, None, None, None, None)
        assert rc != 0, b
        if "kc" in b or "profile" in b:
            st = np.full((S, 6), 7.0); xo = np.full((S, 2), 7.0)
            for fn in (lib.ntm_kf_step, lib.ntm_kf_step_dev):
                rc = fn(mpc._h, 0, a["profile"], S, x0.ctypes.data, uk.ctypes.data, P.ctypes.data, S, kcp,
                        st.ctypes.data, xo.ctypes.data)
                assert rc != 0, b
            assert np.all(st == 7.0) and np.all(xo == 7.0), b
    st = np.full((S, 6), 7.0)
    for args_ in ((0, 0, S, x0.ctypes.data, None, P.ctypes.data, S, KC.ctypes.data, st.ctypes.data, None),   # u NULL
                  (0, 0, S, x0.ctypes.data, uk.ctypes.data, P.ctypes.data, 2, KC.ctypes.data, st.ctypes.data, None),
                  (2, 0, S, x0.ctypes.data, uk.ctypes.data, P.ctypes.data, S, KC.ctypes.data, st.ctypes.data, None)):
        assert lib.ntm_kf_step(mpc._h, *args_) != 0
    assert np.all(st == 7.0)
    assert mpc.launch_count() == before


def test_montecarlo_and_gateways_12_and_13_against_the_c_abi(mpc):
    import torch
    from ntm_mpc import montecarlo, physics
    S, k_sim, seed = 2048, 10, 3
    w_std, v_std = (1e-3, 30.0), (5e-4, 20.0)
    kc = montecarlo.kf_cov_from_std(w_std, v_std)
    kw = dict(plant_sample={"Cw": (0.5, 2.0)}, w_std=w_std, v_std=v_std, noise_seed=9, kf_cov=kc)
    prm, x0, N = physics.batch_params(3, S, seed)
    PP = montecarlo.plant_batch_params(3, S, seed, None, {"Cw": (0.5, 2.0)})
    dw, dv = montecarlo.noise(S, k_sim, w_std, v_std, 9, torch.device("cuda"))
    to_host = lambda t: t.cpu().numpy().reshape(k_sim, 2, S).transpose(2, 0, 1).copy()
    d, v = to_host(dw), to_host(dv)
    for mode in (OFF, REFRESH, FROZEN):
        res = montecarlo.run(config=3, S=S, seed=seed, k_sim=k_sim, handle=mpc, trajectories=True, state_rows=mode,
                             bounds=XB, **kw)
        got = mpc.closed_loop_observed(x0, prm.T.copy(), N, kc, plant_params=PP.T.copy(), w=d, v=v, k_sim=k_sim,
                                       state_rows=mode, xbounds=XB)
        for key in ("xk", "uk", "cost", "status", "xhat"):
            assert same_bits(res[key], got[key]), key
        stats = mpc.mc_stats(got["xk"], got["uk"], got["cost"], got["status"], prm.T.copy(), bounds=XB)
        assert np.allclose(res["stats"], stats, rtol=1e-12, atol=0, equal_nan=True)
        assert np.array_equal(res["stats"][:4], stats[:4])

    from test_mex_gateway import Mock
    mock = Mock()
    Sm = 64
    P = prm.T[:Sm].copy(); PPm = PP.T[:Sm].copy(); xm = x0[:Sm]
    mat = lambda a: np.ascontiguousarray(a).reshape(Sm, -1).T.copy()        # MATLAB layout: one column per scenario
    for mode in (REFRESH, FROZEN):
        ref = mpc.closed_loop_observed(xm, P, N, kc, plant_params=PPm, plant_profile=RK4, w=d[:Sm], v=v[:Sm],
                                       k_sim=k_sim, state_rows=mode, xbounds=XB)
        xk, uk, cost, inner, status, xhat = mock.call(
            "ntm_mpc_batch_perturbed", [xm.T, P.T, N, k_sim, 10, 1e-14, 0, PPm.T, RK4, mat(d[:Sm]), mat(v[:Sm]), mode,
                                        np.array([XB[0], XB[2]]), np.array([XB[1], XB[3]]), kc], nlhs=6)
        assert same_bits(xk, mat(ref["xk"])) and same_bits(uk, mat(ref["uk"])) and same_bits(cost.ravel(), ref["cost"])
        assert same_bits(xhat, mat(ref["xhat"]))
        assert np.array_equal(inner, mat(ref["inner_iters"]).astype(float)) and np.array_equal(status.ravel(), ref["status"])
    # gateway 13: the records travel through MATLAB and back
    state = np.zeros((Sm, 6))
    mst = np.zeros((0, 0))
    u = np.zeros(Sm)
    for k in range(4):
        y = xm + v[:Sm, k]
        ref = mpc.kf_step(state, y, u, P, kc, RK4 | PLANT_C)
        xh, mst = mock.call("ntm_kf_step", [y.T, u[None, :], P.T, kc, mst, RK4 | PLANT_C], nlhs=2)
        assert same_bits(xh, ref.T) and same_bits(mst, state.T)
        u = np.full(Sm, 3e5 * (k + 1))
