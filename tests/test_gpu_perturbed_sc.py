"""The perturbed loop with getWLc's state rows kept (ntm_mpc_closed_loop_perturbed_sc[_dev]) on the GPU (-m gpu).

1. Bit identity with the step-API composition: k_sim x (ntm_mpc_step_sc at x + v_k, ntm_plant_step on the plant's block
   and profile, + d_k), up to and including each scenario's infeasible step, and the NaN / 0 tail after it, on every
   instantiation (one warp literal / dense Gamma, two and four warps literal), both row modes, plant profiles, parameter
   counts, layouts, host and device entries.
2. Nothing perturbed: bit-identical to ntm_mpc_closed_loop_sc, including config 3 at full size with the script's box.
3. STATE_ROWS_OFF is ntm_mpc_closed_loop_perturbed: the same bits and the same kernel.
4. Scenarios stay independent.  5. One launch per call, argument errors launch and copy nothing, the caller's stream.
6. montecarlo.run(state_rows=..., plant_sample=..., w_std=..., v_std=...) and MEX gateway 12 against the C ABI."""

import numpy as np
import pytest

from oracle import ntm_oracle as o
from test_gpu_perturbed import blocks, host_cost, same_bits

pytestmark = pytest.mark.gpu

RHO1_SQ, GAMMA_I, F_XK, PLANT_C, FIXED, DENSE_G, RK4, TAUE_W = 1, 2, 4, 8, 16, 32, 64, 128
PLANT_BITS = RHO1_SQ | PLANT_C | RK4 | TAUE_W
REFRESH, FROZEN = 1, 2
KEYS = ("xk", "uk", "Uk", "inner_iters", "qp_iters", "status")
XB = (0.05, 0.16, 2000.0, 12000.0)          # binds on part of config 3 and is infeasible on another (test_gpu_ext.py)


@pytest.fixture(scope="module")
def mpc():
    import ntm_mpc
    h = ntm_mpc.NtmMpc(0)
    yield h
    h.close()


def noise(S, k_sim, seed=5):
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(S, k_sim, 2)) * np.array([4e-3, 600.0])     # large enough that true states leave the box and
    v = rng.normal(size=(S, k_sim, 2)) * np.array([5e-3, 500.0])     # measurements alone end some scenarios
    return d, v


def composition_sc(mpc, x0, P, N, k_sim, i_sim, eps, profile, PP, pprof, d, v, mode, xb):
    """The contract, written out with the step API: ntm_mpc_step_sc at y_k = x_k + v_k, ntm_plant_step, + d_k; a
    scenario whose step comes back infeasible ends there (NaN u, U and later states, iteration counts 0 after it)."""
    import ntm_mpc
    S = x0.shape[0]
    state = np.zeros((S, ntm_mpc.ctrl_doubles(N)))
    x = x0.copy()
    xk = np.full((S, k_sim + 1, 2), np.nan); xk[:, 0] = x0
    uk = np.full((S, k_sim), np.nan); Uk = np.full((S, k_sim, N), np.nan)
    inner = np.zeros((S, k_sim), dtype=np.int32); qpit = np.zeros((S, k_sim), dtype=np.int32)
    status = np.zeros(S, dtype=np.int32)
    live = np.ones(S, dtype=bool)
    k_inf = np.full(S, -1)
    for k in range(k_sim):
        y = x if v is None else x + v[:, k]
        r = mpc.mpc_step(state, np.where(live[:, None], y, 0.1), P, N, i_sim, eps, profile, want_U=True,
                         state_rows=mode, xbounds=xb)
        inner[live, k] = r["inner_iters"][live]; qpit[live, k] = r["qp_iters"][live]
        status[live] = np.maximum(status[live], r["status"][live])
        bad_y = live & ~np.all(np.isfinite(y), axis=1)
        status[bad_y] = np.maximum(status[bad_y], 2)
        dead = live & (r["status"] == 3)
        k_inf[dead] = k
        live &= ~dead
        xn = mpc.plant_step(x, np.where(live, r["u"], 0.0), PP, pprof)
        if d is not None:
            xn = xn + d[:, k]
        x = np.where(live[:, None], xn, x)
        xk[live, k + 1] = x[live]; uk[live, k] = r["u"][live]; Uk[live, k] = r["U"][live]
    fin = live & ~np.all(np.isfinite(xk[:, -1]), axis=1)
    status[fin] = np.maximum(status[fin], 2)
    return dict(xk=xk, uk=uk, Uk=Uk, inner_iters=inner, qp_iters=qpit, status=status, k_inf=k_inf)


def perturbed_sc_dev(mpc, x0, P, N, k_sim, i_sim, eps, profile, PP, pprof, d, v, layout, mode, xb, stream=None):
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
    Uk = torch.empty(S * N * k_sim, **f64); cost = torch.empty(S, **f64)
    i32 = dict(dtype=torch.int32, device=dev)
    inner = torch.empty(S * k_sim, **i32); qp = torch.empty(S * k_sim, **i32); st = torch.empty(S, **i32)
    torch.cuda.synchronize()
    if stream is not None:
        mpc.set_stream(stream.cuda_stream)
    ptr = lambda t: 0 if t is None else t.data_ptr()
    count = lambda B: B.shape[0] if B.ndim == 2 else 1
    mpc.closed_loop_perturbed_dev(S, N, k_sim, i_sim, eps, profile, layout, ptr(x), ptr(p), count(P),
                                  ptr(pp), count(PP) if PP is not None else 0, pprof,
                                  ptr(dw), ptr(dv), ptr(xk), ptr(uk), ptr(Uk), ptr(cost), ptr(inner), ptr(qp), ptr(st),
                                  state_rows=mode, xbounds=xb)
    if stream is not None:
        stream.synchronize()
        mpc.reset_stream()
    mpc.sync()

    def get(t, E):
        a = t.cpu().numpy()
        return a.reshape(E, S).T.copy() if soa else a.reshape(S, E)
    return dict(xk=get(xk, 2 * (k_sim + 1)).reshape(S, k_sim + 1, 2), uk=get(uk, k_sim),
                Uk=get(Uk, N * k_sim).reshape(S, k_sim, N), cost=cost.cpu().numpy(),
                inner_iters=get(inner, k_sim), qp_iters=get(qp, k_sim), status=st.cpu().numpy())


def outside(x, xb):
    return (x[..., 0] < xb[0]) | (x[..., 0] > xb[1]) | (x[..., 1] < xb[2]) | (x[..., 1] > xb[3])


# N, profile, plant_profile, per-scenario controller block, per-scenario plant block, layout, entry, rows, d / v
CASES = [
    (3, FIXED, 0, False, True, 0, "host", REFRESH, True),
    (10, 0, RK4, True, True, 1, "dev", FROZEN, True),
    (20, FIXED, TAUE_W, True, False, 0, "dev", REFRESH, True),
    (32, 0, PLANT_C, True, True, 0, "host", FROZEN, True),
    (20, FIXED, RHO1_SQ | RK4, True, True, 1, "dev", FROZEN, False),
    (24, GAMMA_I | FIXED, RHO1_SQ, True, True, 0, "dev", REFRESH, True),
    (16, GAMMA_I, RK4, False, True, 1, "dev", FROZEN, True),
    (30, DENSE_G, TAUE_W, True, True, 0, "host", FROZEN, True),
    (20, DENSE_G | FIXED, 0, True, False, 1, "dev", REFRESH, False),
    (40, FIXED, RK4, True, True, 0, "dev", REFRESH, True),
    (64, 0, TAUE_W, True, True, 1, "dev", FROZEN, True),
    (64, FIXED, PLANT_C, True, True, 0, "host", REFRESH, True),
    (100, FIXED, PLANT_C | RK4, True, True, 1, "dev", FROZEN, True),
    (100, 0, 0, True, False, 0, "host", FROZEN, True),
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
    ref = composition_sc(mpc, x0, P, N, k_sim, i_sim, eps, profile, PP, pprof, d, v, mode, XB)
    if entry == "host":
        got = mpc.closed_loop_perturbed(x0, P, N, plant_params=PP, plant_profile=pprof, w=d, v=v, k_sim=k_sim,
                                        i_sim=i_sim, eps=eps, profile=profile, want_Uk=True, state_rows=mode, xbounds=XB)
    else:
        got = perturbed_sc_dev(mpc, x0, P, N, k_sim, i_sim, eps, profile, PP, pprof, d, v, layout, mode, XB)
    for key in KEYS:
        assert same_bits(got[key], ref[key]), key
    ended = ref["k_inf"] >= 0
    assert np.all(np.isnan(got["cost"][ended]))
    assert np.allclose(got["cost"][~ended], host_cost(got["xk"][~ended], np.broadcast_to(P, (S, P.shape[-1]))[~ended]),
                       rtol=1e-13, atol=0)
    # what the sample must contain: scenarios that turn infeasible, ones the rows steer off the box-QP answer, ...
    box = mpc.closed_loop_perturbed(x0, P, N, plant_params=PP, plant_profile=pprof, w=d, v=v, k_sim=k_sim, i_sim=i_sim,
                                    eps=eps, profile=profile)
    assert np.any(ended)
    fin = np.isfinite(got["uk"])
    assert np.any(fin & (got["uk"] != box["uk"]))
    # ... one whose true state leaves the box (after the start) ...
    assert np.any(outside(got["xk"][:, 1:], XB) & np.all(np.isfinite(got["xk"][:, 1:]), axis=-1))
    if v is not None:
        # ... and one ended by its measurement: y_k outside the box while x_k was inside
        s_end = np.nonzero(ended)[0]
        xs = got["xk"][s_end, ref["k_inf"][s_end]]
        ys = xs + v[s_end, ref["k_inf"][s_end]]
        assert np.any(outside(ys, XB) & ~outside(xs, XB))


# nothing perturbed, every EXT 4 instantiation: config 3 at full size with the script's box in both modes
UNPERTURBED = [(3, None, 20, 0, REFRESH, None), (3, None, 20, FIXED, FROZEN, None), (3, 512, 10, RK4, REFRESH, XB),
               (3, 512, 24, GAMMA_I, FROZEN, XB), (3, 512, 30, DENSE_G | FIXED, REFRESH, XB),
               (3, 512, 20, RK4 | RHO1_SQ | PLANT_C, FROZEN, XB), (3, 256, 48, 0, FROZEN, XB),
               (3, 256, 100, FIXED | RK4, REFRESH, XB)]


@pytest.mark.parametrize("cfg,S,N,profile,mode,xb", UNPERTURBED,
                         ids=[f"cfg{c[0]}-S{c[1]}-N{c[2]}-p{c[3]}-r{c[4]}" for c in UNPERTURBED])
def test_no_perturbation_is_the_state_row_loop(mpc, cfg, S, N, profile, mode, xb):
    phys, x0, _ = o.make_batch(cfg, S=S)
    P = o.derive_params_batch(phys).T.copy()
    ref = mpc.closed_loop(x0, P, N, profile=profile, want_Uk=True, state_rows=mode, xbounds=xb)
    got = mpc.closed_loop_perturbed(x0, P, N, profile=profile, want_Uk=True, state_rows=mode, xbounds=xb)
    for key in KEYS + ("cost",):
        assert same_bits(got[key], ref[key]), key


def test_rows_off_is_the_box_qp_perturbed_loop_and_its_kernel(mpc):
    from torch.profiler import ProfilerActivity, profile
    S, N, k_sim = 48, 20, 6
    P, PP, x0 = blocks(S)
    d, v = noise(S, k_sim)
    kw = dict(plant_params=PP, plant_profile=RK4, w=d, v=v, k_sim=k_sim, want_Uk=True)
    import ntm_mpc
    names = []
    for mode in (None, 0, REFRESH):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            if mode is None:                     # the box-QP entry itself
                r = mpc.closed_loop_perturbed(x0, P, N, **kw)
            else:
                r = perturbed_sc_dev(mpc, x0, P, N, k_sim, 10, 1e-14, 0, PP, RK4, d, v, ntm_mpc.LAYOUT_MATLAB, mode, XB)
        names.append(sorted({e.name for e in prof.events() if "closed_loop_kernel" in e.name}))
        if mode is None:
            base = r
        elif mode == 0:
            for key in KEYS + ("cost",):
                assert same_bits(r[key], base[key]), key
    assert len(names[0]) == 1 and names[1] == names[0], names
    assert names[2] != names[0], names


def test_scenarios_stay_independent(mpc):
    S, N, k_sim = 32, 20, 8
    P, PP, x0 = blocks(S)
    d, v = noise(S, k_sim)
    kw = dict(plant_profile=RK4, k_sim=k_sim, state_rows=FROZEN, xbounds=XB)
    base = mpc.closed_loop_perturbed(x0, P, N, plant_params=PP, w=d, v=v, **kw)
    v2 = v.copy()
    v2[9, 2, 1] = np.nan
    got = mpc.closed_loop_perturbed(x0, P, N, plant_params=PP, w=d, v=v2, **kw)
    keep = np.setdiff1d(np.arange(S), [9])
    for key in ("xk", "uk", "cost", "inner_iters", "qp_iters", "status"):
        assert same_bits(got[key][keep], base[key][keep]), key
    assert got["status"][9] >= 2
    perm = np.random.default_rng(4).permutation(S)
    pg = mpc.closed_loop_perturbed(x0[perm], P[perm], N, plant_params=PP[perm], w=d[perm], v=v[perm], **kw)
    for key in ("xk", "uk", "cost", "inner_iters", "qp_iters", "status"):
        assert same_bits(pg[key], base[key][perm]), key


def test_one_launch_argument_errors_and_the_callers_stream(mpc):
    import torch
    import ntm_mpc
    S, N, k_sim = 16, 12, 5
    P, PP, x0 = blocks(S)
    d, v = noise(S, k_sim)
    args = (mpc, x0, P, N, k_sim, 10, 1e-14, 0, PP, RK4, d, v, 0, REFRESH, XB)
    ref = perturbed_sc_dev(*args)
    before = mpc.launch_count()
    perturbed_sc_dev(*args)
    assert mpc.launch_count() == before + 1
    s = torch.cuda.Stream()
    got = perturbed_sc_dev(*args, stream=s)
    for key in KEYS + ("cost",):
        assert same_bits(got[key], ref[key]), key
    # argument errors, through the C entries themselves (the Python front end refuses some of them first): nothing
    # launched, nothing copied (the host entry's output arrays stay as they were)
    before = mpc.launch_count()
    bad = [dict(profile=TAUE_W), dict(plant_profile=GAMMA_I), dict(state_rows=3), dict(state_rows=-1),
           dict(xbounds=np.array([0.16, 0.05, 2000.0, 12000.0])), dict(xbounds=np.array([0.05, 0.16, np.nan, 1.0])),
           dict(xbounds=None), dict(profile=GAMMA_I, N=40), dict(profile=DENSE_G, N=33), dict(N=129), dict(ppc=2)]
    lib = mpc._lib
    for b in bad:
        a = dict(profile=0, plant_profile=RK4, state_rows=REFRESH, xbounds=np.array(XB), N=N, ppc=S)
        a.update(b)
        xb = None if a["xbounds"] is None else a["xbounds"].ctypes.data
        xk = np.full((S, k_sim + 1, 2), 7.0); uk = np.full((S, k_sim), 7.0)
        rc = lib.ntm_mpc_closed_loop_perturbed_sc(mpc._h, ntm_mpc.LAYOUT_MATLAB, a["profile"], S, a["N"], k_sim, 10,
                                                  1e-14, x0.ctypes.data, P.ctypes.data, S, a["state_rows"], xb,
                                                  PP.ctypes.data, a["ppc"], a["plant_profile"], d.ctypes.data,
                                                  v.ctypes.data, xk.ctypes.data, uk.ctypes.data, None, None, None,
                                                  None, None)
        assert rc != 0, b
        assert np.all(xk == 7.0) and np.all(uk == 7.0), b
        rc = lib.ntm_mpc_closed_loop_perturbed_sc_dev(mpc._h, 0, a["profile"], S, a["N"], k_sim, 10, 1e-14, 1, 1, 1,
                                                      a["state_rows"], xb, 1, a["ppc"], a["plant_profile"], None, None,
                                                      1, 1, None, None, None, None, None)
        assert rc != 0, b
    assert mpc.launch_count() == before


def test_montecarlo_and_gateway_12_against_the_c_abi(mpc):
    import torch
    from ntm_mpc import montecarlo, physics
    S, k_sim, seed = 2048, 10, 3
    kw = dict(plant_sample={"Cw": (0.5, 2.0)}, w_std=(1e-3, 30.0), v_std=(5e-4, 20.0), noise_seed=9)
    for mode in (REFRESH, FROZEN):
        res = montecarlo.run(config=3, S=S, seed=seed, k_sim=k_sim, handle=mpc, trajectories=True, state_rows=mode,
                             bounds=XB, **kw)
        prm, x0, N = physics.batch_params(3, S, seed)
        PP = montecarlo.plant_batch_params(3, S, seed, None, {"Cw": (0.5, 2.0)})
        dw, dv = montecarlo.noise(S, k_sim, (1e-3, 30.0), (5e-4, 20.0), 9, torch.device("cuda"))
        to_host = lambda t: t.cpu().numpy().reshape(k_sim, 2, S).transpose(2, 0, 1).copy()
        d, v = to_host(dw), to_host(dv)
        got = mpc.closed_loop_perturbed(x0, prm.T.copy(), N, plant_params=PP.T.copy(), w=d, v=v, k_sim=k_sim,
                                        state_rows=mode, xbounds=XB)
        for key in ("xk", "uk", "cost", "status"):
            assert same_bits(res[key], got[key]), key
        stats = mpc.mc_stats(got["xk"], got["uk"], got["cost"], got["status"], prm.T.copy(), bounds=XB)
        assert np.allclose(res["stats"], stats, rtol=1e-12, atol=0, equal_nan=True)
        assert np.array_equal(res["stats"][:4], stats[:4])
        assert stats[3] > 0                                          # infeasible scenarios are counted

    from test_mex_gateway import Mock
    mock = Mock()
    Sm = 64
    P = prm.T[:Sm].copy(); PPm = PP.T[:Sm].copy(); xm = x0[:Sm]
    mat = lambda a: np.ascontiguousarray(a).reshape(Sm, -1).T.copy()        # MATLAB layout: one column per scenario
    for mode in (REFRESH, FROZEN):
        ref = mpc.closed_loop_perturbed(xm, P, N, plant_params=PPm, plant_profile=RK4, w=d[:Sm], v=v[:Sm], k_sim=k_sim,
                                        state_rows=mode, xbounds=XB)
        xk, uk, cost, inner, status = mock.call(
            "ntm_mpc_batch_perturbed", [xm.T, P.T, N, k_sim, 10, 1e-14, 0, PPm.T, RK4, mat(d[:Sm]), mat(v[:Sm]), mode,
                                        np.array([XB[0], XB[2]]), np.array([XB[1], XB[3]])], nlhs=5)
        assert same_bits(xk, mat(ref["xk"])) and same_bits(uk, mat(ref["uk"])) and same_bits(cost.ravel(), ref["cost"])
        assert np.array_equal(inner, mat(ref["inner_iters"]).astype(float)) and np.array_equal(status.ravel(), ref["status"])
