"""The fused loop against a perturbed plant (ntm_mpc_closed_loop_perturbed[_dev]) on the GPU (-m gpu).

1. Bit identity with the step-API composition: k_sim x (ntm_mpc_step at x + v_k, ntm_plant_step on the plant's block
   and profile, + d_k), on every box-QP instantiation (one warp literal / dense, multi-warp dense, long tableau in
   registers and in shared memory), plant profiles, parameter counts, layouts, host and device entries.
2. No perturbation: bit-identical to ntm_mpc_closed_loop, including config 3 at full size (two-phase reference).
3. Scenarios stay independent.  4. One launch per call, argument errors launch nothing, the caller's stream.
5. montecarlo.run(plant_sample=..., w_std=..., v_std=...) and MEX gateway 12 against the C ABI."""

import numpy as np
import pytest

from oracle import ntm_oracle as o

pytestmark = pytest.mark.gpu

RHO1_SQ, GAMMA_I, F_XK, PLANT_C, FIXED, DENSE_G, RK4, TAUE_W = 1, 2, 4, 8, 16, 32, 64, 128
CONS = GAMMA_I | F_XK | PLANT_C
PLANT_BITS = RHO1_SQ | PLANT_C | RK4 | TAUE_W
KEYS = ("xk", "uk", "Uk", "inner_iters", "qp_iters", "status")


@pytest.fixture(scope="module")
def mpc():
    import ntm_mpc
    h = ntm_mpc.NtmMpc(0)
    yield h
    h.close()


def blocks(S, seed=11):
    """Controller block (config 3 draws), plant block (the same with Cw and c_tauE drawn anew), x0."""
    phys, x0, _ = o.make_batch(3, S=S, seed=seed)
    pphys, _, _ = o.make_batch(3, S=S, seed=seed, sample={"Cw": (0.5, 2.0), "c_tauE": (0.0, 1.5)})
    return o.derive_params_batch(phys).T.copy(), o.derive_params_batch(pphys).T.copy(), x0


def noise(S, k_sim, seed=5):
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(S, k_sim, 2)) * np.array([1e-3, 40.0])
    v = rng.normal(size=(S, k_sim, 2)) * np.array([1e-3, 40.0])
    return d, v


def composition(mpc, x0, P, N, k_sim, i_sim, eps, profile, PP, pprof, d, v):
    """The contract, written out with the step API: ntm_mpc_step at y_k = x_k + v_k, ntm_plant_step, + d_k."""
    import ntm_mpc
    S = x0.shape[0]
    state = np.zeros((S, ntm_mpc.ctrl_doubles(N)))
    x, xs, us, Us, inn, qps = x0.copy(), [x0.copy()], [], [], [], []
    status = np.zeros(S, dtype=np.int32)
    for k in range(k_sim):
        y = x if v is None else x + v[:, k]
        r = mpc.mpc_step(state, y, P, N, i_sim, eps, profile, want_U=True)
        x = mpc.plant_step(x, r["u"], PP, pprof)
        if d is not None:
            x = x + d[:, k]
        xs.append(x); us.append(r["u"]); Us.append(r["U"]); inn.append(r["inner_iters"]); qps.append(r["qp_iters"])
        status = np.maximum(status, r["status"])
        status[~np.all(np.isfinite(y), axis=1)] = np.maximum(status[~np.all(np.isfinite(y), axis=1)], 2)
    xk = np.stack(xs, 1)
    status[~np.all(np.isfinite(xk[:, -1]), axis=1)] = np.maximum(status[~np.all(np.isfinite(xk[:, -1]), axis=1)], 2)
    return dict(xk=xk, uk=np.stack(us, 1), Uk=np.stack(Us, 1), inner_iters=np.stack(inn, 1), qp_iters=np.stack(qps, 1),
                status=status)


def host_cost(xk, P):
    P = np.broadcast_to(P, (xk.shape[0], P.shape[-1]))
    e1, e2 = xk[:, 1:, 0] - P[:, 10, None], xk[:, 1:, 1] - P[:, 11, None]
    return np.sum(e1 * (P[:, 12, None] * e1 + P[:, 13, None] * e2) + e2 * (P[:, 13, None] * e1 + P[:, 14, None] * e2), axis=1)


def perturbed_dev(mpc, x0, P, N, k_sim, i_sim, eps, profile, PP, pprof, d, v, layout, stream=None):
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
                                  ptr(dw), ptr(dv), ptr(xk), ptr(uk), ptr(Uk), ptr(cost), ptr(inner), ptr(qp), ptr(st))
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


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype.kind == "f":
        return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))
    return np.array_equal(a, b)


# N, profile, plant_profile, per-scenario controller block, per-scenario plant block, layout, entry
CASES = [
    (8, FIXED, 0, False, True, 0, "host"),
    (20, 0, RK4, True, True, 1, "dev"),
    (24, GAMMA_I, TAUE_W, True, False, 0, "dev"),
    (16, CONS | FIXED, PLANT_C, False, True, 0, "host"),
    (30, DENSE_G, RHO1_SQ, True, True, 1, "dev"),
    (32, 0, RK4 | TAUE_W, True, True, 0, "host"),
    (48, 0, RK4 | TAUE_W, True, True, 0, "dev"),
    (64, GAMMA_I | FIXED, TAUE_W, True, False, 1, "dev"),
    (80, FIXED, RK4, False, True, 0, "host"),
    (100, CONS, RK4, True, True, 1, "dev"),
    (104, 0, PLANT_C, True, True, 1, "dev"),
    (110, FIXED, 0, True, False, 0, "dev"),
    (128, 0, RK4, True, True, 1, "host"),
    (12, RHO1_SQ, RK4 | RHO1_SQ, True, True, 0, "dev"),
    (72, RHO1_SQ | FIXED, RK4 | RHO1_SQ | PLANT_C, True, True, 1, "host"),
]


@pytest.mark.parametrize("N,profile,pprof,pc_s,ppc_s,layout,entry", CASES,
                         ids=[f"N{c[0]}-p{c[1]}-pp{c[2]}-{c[6]}-L{c[5]}" for c in CASES])
def test_bit_identical_to_the_step_composition(mpc, N, profile, pprof, pc_s, ppc_s, layout, entry):
    S, k_sim, i_sim, eps = 24, 6, 10, 1e-14
    P, PP, x0 = blocks(S)
    if not pc_s:
        P = P[0]
    if not ppc_s:
        PP = PP[3]
    d, v = noise(S, k_sim)
    ref = composition(mpc, x0, P, N, k_sim, i_sim, eps, profile, PP, pprof, d, v)
    if entry == "host":
        got = mpc.closed_loop_perturbed(x0, P, N, plant_params=PP, plant_profile=pprof, w=d, v=v, k_sim=k_sim,
                                        i_sim=i_sim, eps=eps, profile=profile, want_Uk=True)
    else:
        got = perturbed_dev(mpc, x0, P, N, k_sim, i_sim, eps, profile, PP, pprof, d, v, layout)
    for key in KEYS:
        assert same_bits(got[key], ref[key]), key
    assert np.allclose(got["cost"], host_cost(got["xk"], P), rtol=1e-13, atol=0)
    # the perturbation reached the controller (or, where every input of the sample sits on the box, at least the plant)
    plain = mpc.closed_loop(x0, P, N, k_sim=k_sim, i_sim=i_sim, eps=eps, profile=profile)
    Pb = np.broadcast_to(P, (S, P.shape[-1]))
    on_box = np.all((plain["uk"] == Pb[:, 8, None]) | (plain["uk"] == Pb[:, 9, None]))
    assert np.any(got["uk"] != plain["uk"]) or (on_box and np.any(got["xk"] != plain["xk"]))


# every box-QP instantiation, unperturbed: config 3 at full size takes the two-phase launch in the reference arm
UNPERTURBED = [(3, None, 20, 0), (2, 512, 24, GAMMA_I | FIXED), (2, 512, 10, RK4), (2, 512, 30, CONS),
               (5, 256, 48, 0), (5, 256, 64, DENSE_G), (5, 256, 100, FIXED | RK4 | PLANT_C), (5, 256, 110, 0),
               (5, 256, 96, CONS), (2, 512, 20, RK4 | RHO1_SQ), (5, 256, 64, RK4 | RHO1_SQ | PLANT_C),
               (5, 256, 100, RK4 | RHO1_SQ)]


@pytest.mark.parametrize("cfg,S,N,profile", UNPERTURBED, ids=[f"cfg{c[0]}-N{c[2]}-p{c[3]}" for c in UNPERTURBED])
def test_no_perturbation_is_the_fused_loop(mpc, cfg, S, N, profile):
    phys, x0, _ = o.make_batch(cfg, S=S)
    P = o.derive_params_batch(phys).T.copy()
    ref = mpc.closed_loop(x0, P, N, profile=profile, want_Uk=True)
    got = mpc.closed_loop_perturbed(x0, P, N, profile=profile, want_Uk=True)
    got2 = mpc.closed_loop_perturbed(x0, P, N, plant_params=P, plant_profile=profile & PLANT_BITS, profile=profile)
    for key in KEYS + ("cost",):
        assert same_bits(got[key], ref[key]), key
        if key != "Uk":
            assert same_bits(got2[key], ref[key]), key


def test_scenarios_stay_independent(mpc):
    S, N, k_sim = 32, 20, 8
    P, PP, x0 = blocks(S)
    d, v = noise(S, k_sim)
    base = mpc.closed_loop_perturbed(x0, P, N, plant_params=PP, plant_profile=RK4, w=d, v=v, k_sim=k_sim)
    d2, v2, PP2 = d.copy(), v.copy(), PP.copy()
    d2[5, 3] *= 3.0
    v2[9, 2, 1] = np.nan
    PP2[12, 1] *= 1.5
    got = mpc.closed_loop_perturbed(x0, P, N, plant_params=PP2, plant_profile=RK4, w=d2, v=v2, k_sim=k_sim)
    keep = np.setdiff1d(np.arange(S), [5, 9, 12])
    for key in ("xk", "uk", "cost", "inner_iters", "qp_iters", "status"):
        assert same_bits(got[key][keep], base[key][keep]), key
    for s in (5, 9, 12):
        assert not same_bits(got["xk"][s], base["xk"][s]), s
    assert got["status"][9] == 2 and np.all(np.isnan(got["xk"][9, -1]))


def test_one_launch_argument_errors_and_the_callers_stream(mpc):
    import torch
    import ntm_mpc
    S, N, k_sim = 16, 12, 5
    P, PP, x0 = blocks(S)
    d, v = noise(S, k_sim)
    ref = perturbed_dev(mpc, x0, P, N, k_sim, 10, 1e-14, 0, PP, RK4, d, v, 0)
    before = mpc.launch_count()
    perturbed_dev(mpc, x0, P, N, k_sim, 10, 1e-14, 0, PP, RK4, d, v, 0)
    assert mpc.launch_count() == before + 1
    s = torch.cuda.Stream()
    got = perturbed_dev(mpc, x0, P, N, k_sim, 10, 1e-14, 0, PP, RK4, d, v, 0, stream=s)
    for key in KEYS + ("cost",):
        assert same_bits(got[key], ref[key]), key
    before = mpc.launch_count()
    for kw in (dict(profile=TAUE_W), dict(plant_profile=GAMMA_I), dict(plant_profile=F_XK)):
        args = dict(profile=0, plant_profile=0)
        args.update(kw)
        with pytest.raises(ntm_mpc.NtmError):
            mpc.closed_loop_perturbed_dev(S, N, k_sim, 10, 1e-14, args["profile"], 0, 1, 1, 1, 0, 0,
                                          args["plant_profile"], 0, 0, 1, 1)
    with pytest.raises(ntm_mpc.NtmError):                            # plant_params_count neither 1 nor S
        mpc.closed_loop_perturbed_dev(S, N, k_sim, 10, 1e-14, 0, 0, 1, 1, 1, 1, 2, 0, 0, 0, 1, 1)
    with pytest.raises(ntm_mpc.NtmError):                            # NULL x0
        mpc.closed_loop_perturbed_dev(S, N, k_sim, 10, 1e-14, 0, 0, 0, 1, 1, 0, 0, 0, 0, 0, 1, 1)
    with pytest.raises(ntm_mpc.NtmError):                            # N out of range
        mpc.closed_loop_perturbed_dev(S, 129, k_sim, 10, 1e-14, 0, 0, 1, 1, 1, 0, 0, 0, 0, 0, 1, 1)
    assert mpc.launch_count() == before


def test_montecarlo_and_gateway_12_against_the_c_abi(mpc):
    import torch
    import ntm_mpc
    from ntm_mpc import montecarlo, physics
    S, k_sim, seed = 2048, 10, 3
    res = montecarlo.run(config=3, S=S, seed=seed, k_sim=k_sim, handle=mpc, trajectories=True,
                         plant_sample={"Cw": (0.5, 2.0)}, plant_profile=RK4, w_std=(1e-3, 30.0), v_std=(5e-4, 20.0),
                         noise_seed=9)
    prm, x0, N = physics.batch_params(3, S, seed)
    PP = montecarlo.plant_batch_params(3, S, seed, None, {"Cw": (0.5, 2.0)})
    dw, dv = montecarlo.noise(S, k_sim, (1e-3, 30.0), (5e-4, 20.0), 9, torch.device("cuda"))
    to_host = lambda t: t.cpu().numpy().reshape(k_sim, 2, S).transpose(2, 0, 1).copy()
    d, v = to_host(dw), to_host(dv)
    got = mpc.closed_loop_perturbed(x0, prm.T.copy(), N, plant_params=PP.T.copy(), plant_profile=RK4, w=d, v=v,
                                    k_sim=k_sim)
    for key in ("xk", "uk", "cost", "status"):
        assert same_bits(res[key], got[key]), key
    stats = mpc.mc_stats(got["xk"], got["uk"], got["cost"], got["status"], prm.T.copy())
    assert np.allclose(res["stats"], stats, rtol=1e-12, atol=0) and np.array_equal(res["stats"][:4], stats[:4])
    assert np.any(res["uk"] != montecarlo.run(config=3, S=S, seed=seed, k_sim=k_sim, handle=mpc, trajectories=True)["uk"])

    from test_mex_gateway import Mock
    mock = Mock()
    Sm = 64
    P = prm.T[:Sm].copy(); PPm = PP.T[:Sm].copy(); xm = x0[:Sm]
    ref = mpc.closed_loop_perturbed(xm, P, N, plant_params=PPm, plant_profile=RK4, w=d[:Sm], v=v[:Sm], k_sim=k_sim)
    mat = lambda a: np.ascontiguousarray(a).reshape(Sm, -1).T.copy()        # MATLAB layout: one column per scenario
    xk, uk, cost, inner, status = mock.call("ntm_mpc_batch_perturbed",
                                            [xm.T, P.T, N, k_sim, 10, 1e-14, 0, PPm.T, RK4, mat(d[:Sm]), mat(v[:Sm])],
                                            nlhs=5)
    assert same_bits(xk, mat(ref["xk"])) and same_bits(uk, mat(ref["uk"])) and same_bits(cost.ravel(), ref["cost"])
    assert np.array_equal(inner, mat(ref["inner_iters"]).astype(float)) and np.array_equal(status.ravel(), ref["status"])
    mock.workspace({})
    xk0 = mock.call("ntm_mpc_batch_perturbed", [xm.T, P.T, N, k_sim, 10, 1e-14, 0, np.zeros((0, 0)), 0,
                                                np.zeros((0, 0)), np.zeros((0, 0))], nlhs=1)[0]
    assert same_bits(xk0, mat(mpc.closed_loop(xm, P, N, k_sim=k_sim)["xk"]))
