"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI (ctypes -> libntm_mpc.so), against the
oracle on the same seeded inputs, against the committed golden fixtures, and -- at BASELINE.json's
full sizes -- through size-independent properties.

Tolerances (north star): 1e-10 relative on Phi/Gamma/Lambda, 1e-6 relative on the EC-power and
island-width trajectories, measured as max|d| / max(||ref||_inf, floor) per quantity (a floor is
needed because in the default scenario w sits at 1e-18 noise).
"""
import math
import os

import numpy as np
import pytest

from oracle import c_oracle as co
from oracle import ntm_oracle as o

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")
TOL_COND = 1e-10
TOL_TRAJ = 1e-6


@pytest.fixture(scope="module")
def mpc():
    import ntm_mpc
    h = ntm_mpc.NtmMpc(0)
    yield h
    h.close()


def rel(a, b, floor=0.0):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), floor, 1e-300))


def traj_err(g_uk, g_xk, c_uk, c_xk, umax):
    """per-scenario relative errors of the EC power and island-width trajectories"""
    du = np.max(np.abs(g_uk - c_uk), axis=1) / umax
    w = c_xk[:, :, 0]
    dw = np.max(np.abs(g_xk[:, :, 0] - w), axis=1) / np.maximum(np.max(np.abs(w), axis=1), 1e-3)
    om = c_xk[:, :, 1]
    dom = np.max(np.abs(g_xk[:, :, 1] - om), axis=1) / np.maximum(np.max(np.abs(om), axis=1), 1.0)
    return du, dw, dom


def sample_states(S, seed):
    rng = np.random.default_rng(seed)
    return np.column_stack([rng.uniform(0.0, 0.2, S), rng.uniform(300.0, 30000.0, S)])


# ------------------------------------------------------------------ device sanity
def test_device_is_blackwell_and_library_is_native(mpc):
    info = mpc.device_info()
    assert info["cc_major"] == 10, info
    assert info["sm_count"] >= 100
    before = mpc.launch_count()
    mpc.rho(np.array([[0.08, 6000.0]]), o.derive_params(o.default_physics()))
    assert mpc.launch_count() == before + 1


# ------------------------------------------------------------------ rho1.m, rho2.m, rho3.m, A.m, B.m, plant
@pytest.mark.parametrize("variant", [o.RHO1_LIN, o.RHO1_SQ])
def test_rho_and_lpv_match_oracle(mpc, variant):
    phys, _, _ = o.make_batch(3, S=512)
    P = o.derive_params_batch(phys)
    X = sample_states(512, 3)
    r1, r2, r3 = mpc.rho(X, P.T, profile=variant)
    A, B = mpc.lpv_AB(r1, r2, r3, P.T)
    for s in range(0, 512, 7):
        p = o.scenario(phys, s)
        e1, e2, e3 = o.rho1(X[s], p["w_marg"], variant), o.rho2(X[s]), o.rho3(X[s], p["w_dep"])
        assert r1[s] == pytest.approx(e1, rel=1e-14) and r2[s] == pytest.approx(e2, rel=1e-14)
        assert r3[s] == pytest.approx(e3, rel=1e-14)
        Af, Bf, _ = o.model_callables(p)
        assert rel(A[s], Af(e1, e2)) < 1e-14 and rel(B[s], Bf(e3)) < 1e-14
        assert A[s][0, 1] == 0.0 and B[s][1] == 0.0


def test_rho_ieee_special_values(mpc):
    p = o.derive_params(o.default_physics())
    X = np.array([[0.08, 0.0], [0.0, 0.0], [-0.0158, 5000.0], [np.nan, 1.0]])
    r1, r2, r3 = mpc.rho(X, p)
    assert np.isinf(r2[0]) and np.isnan(r2[1])                   # w^2/0, 0/0 (rho2.m:2)
    with np.errstate(all="ignore"):
        assert r3[2] == pytest.approx(o.rho3(X[2], 0.024), rel=1e-9)     # near the pole of rho3.m:3
    assert np.isnan(r1[3]) and np.isnan(r3[3])


@pytest.mark.parametrize("prof", [o.LITERAL, o.CONSISTENT])
def test_plant_step_matches_oracle(mpc, prof):
    phys, _, _ = o.make_batch(4, S=256)
    P = o.derive_params_batch(phys)
    X = sample_states(256, 5)
    u = np.random.default_rng(6).uniform(0, 2e6, 256)
    xn = mpc.plant_step(X, u, P.T, profile=prof.flags())
    for s in range(0, 256, 5):
        p = o.scenario(phys, s)
        Af, Bf, C = o.model_callables(p)
        e = Af(o.rho1(X[s], p["w_marg"]), o.rho2(X[s])) @ X[s] + Bf(o.rho3(X[s], p["w_dep"])) * u[s]
        if prof.plant_affine:
            e = e + C
        assert rel(xn[s], e) < 1e-13


# ------------------------------------------------------------------ Rho_to_PhiGammaLambda.m
def _rho_batch(phys, S, N, seed):
    rng = np.random.default_rng(seed)
    R1 = np.zeros((S, N)); R2 = np.zeros((S, N)); R3 = np.zeros((S, N))
    for s in range(S):
        p = o.scenario(phys, s)
        for i in range(N):
            x = np.array([rng.uniform(0.04, 0.16), rng.uniform(500.0, 14000.0)])
            R1[s, i], R2[s, i], R3[s, i] = o.rho1(x, p["w_marg"]), o.rho2(x), o.rho3(x, p["w_dep"])
    return R1, R2, R3


@pytest.mark.parametrize("N", [1, 2, 3, 10, 20, 32, 33, 64, 65, 100, 128])
@pytest.mark.parametrize("gi", [0, 1])
def test_condense_matches_oracle(mpc, N, gi):
    S = 6
    phys, _, _ = o.make_batch(3, S=S)
    P = o.derive_params_batch(phys)
    R1, R2, R3 = _rho_batch(phys, S, N, 100 + N)
    flags = o.Profile(gamma_index=gi).flags()
    Phi, Gam, Lam = mpc.condense(R1, R2, R3, P.T, profile=flags)
    for s in range(S):
        Af, Bf, C = o.model_callables(o.scenario(phys, s))
        ePhi, eGam, eLam = o.Rho_to_PhiGammaLambda(R1[s], R2[s], R3[s], Af, Bf, C, gi)
        assert rel(Phi[s], ePhi) < TOL_COND
        assert rel(Gam[s], eGam) < TOL_COND
        assert rel(Lam[s], eLam) < TOL_COND
        # exact structure: zeros above the block diagonal, B_j on it
        for j in range(N):
            assert np.all(Gam[s][:2 * j, j] == 0.0)
            assert Gam[s][2 * j + 1, j] == 0.0
        assert np.all(Phi[s][0::2, 1] == 0.0)


@pytest.mark.parametrize("N,prof", [(20, 0), (20, 2), (1, 0), (33, 0), (100, 2)])
def test_condense_soa_layout_is_the_same_numbers(mpc, N, prof):
    """layout flag only permutes storage: run the SoA entry (one thread per scenario) through torch device buffers"""
    import torch
    import ntm_mpc
    S = 37
    phys, _, _ = o.make_batch(3, S=S)
    P = o.derive_params_batch(phys)
    R1, R2, R3 = _rho_batch(phys, S, N, 9)
    Phi, Gam, Lam = mpc.condense(R1, R2, R3, P.T, profile=prof)
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    r1, r2, r3, pp = t(R1.T), t(R2.T), t(R3.T), t(P)                    # SoA: element-major, scenario fastest
    phi = torch.empty(4 * N * S, dtype=torch.float64, device=dev)
    gam = torch.empty(2 * N * N * S, dtype=torch.float64, device=dev)
    lam = torch.empty(2 * N * S, dtype=torch.float64, device=dev)
    mpc.set_stream(torch.cuda.current_stream().cuda_stream)
    mpc.condense_dev(S, N, prof, ntm_mpc.LAYOUT_SOA, r1.data_ptr(), r2.data_ptr(), r3.data_ptr(), pp.data_ptr(), S,
                     phi.data_ptr(), gam.data_ptr(), lam.data_ptr())
    torch.cuda.synchronize()
    mpc.reset_stream()
    g = gam.cpu().numpy().reshape(N, 2 * N, S)                           # [col, row, s]
    # the MATLAB-layout paths are the warp-scan / staged kernels, the SoA path the serial recurrence: same numbers to rounding
    assert rel(g.transpose(2, 1, 0), Gam) < 1e-12
    assert rel(phi.cpu().numpy().reshape(2, 2 * N, S).transpose(2, 1, 0), Phi) < 1e-12
    assert rel(lam.cpu().numpy().reshape(2 * N, S).T, Lam) < 1e-12
    assert np.array_equal(g.transpose(2, 1, 0) == 0.0, Gam == 0.0)       # identical zero pattern
    # and against the oracle directly
    Af, Bf, C = o.model_callables(o.scenario(phys, 3))
    Po, Go, Lo = o.Rho_to_PhiGammaLambda(R1[3], R2[3], R3[3], Af, Bf, C, 1 if prof & 2 else 0)
    assert rel(g[:, :, 3].T, Go) < TOL_COND and rel(lam.cpu().numpy().reshape(2 * N, S)[:, 3], Lo) < TOL_COND


# ------------------------------------------------------------------ G, F
@pytest.mark.parametrize("N", [1, 3, 7, 8, 10, 16, 20, 24, 31, 32, 33, 47, 64, 100, 104, 111, 120, 128])
def test_hessian_grad_matches_oracle(mpc, N):
    S = 5
    phys, _, _ = o.make_batch(3, S=S)
    phys["q12"] = np.full(S, 0.3); phys["q22"] = np.full(S, 2.5)
    P = o.derive_params_batch(phys)
    R1, R2, R3 = _rho_batch(phys, S, N, 200 + N)
    X = sample_states(S, 11)
    Phi = np.zeros((S, 2 * N, 2)); Gam = np.zeros((S, 2 * N, N)); Lam = np.zeros((S, 2 * N))
    exp = []
    for s in range(S):
        p = o.scenario(phys, s)
        Af, Bf, C = o.model_callables(p)
        Phi[s], Gam[s], Lam[s] = o.Rho_to_PhiGammaLambda(R1[s], R2[s], R3[s], Af, Bf, C, s % 2)
        if s == 0:
            Gam[s] += np.random.default_rng(1).standard_normal(Gam[s].shape) * 1e-9    # dense, no structure
        Q = np.array([[p["q11"], p["q12"]], [p["q12"], p["q22"]]])
        exp.append(o.hessian_grad(Phi[s], Gam[s], Lam[s], X[s], [p["r1"], p["r2"]], Q))
    G, F = mpc.hessian_grad(Phi, Gam, Lam, X, P.T)
    for s in range(S):
        assert rel(G[s], exp[s][0]) < TOL_COND
        assert rel(F[s], exp[s][1]) < 1e-9
        assert np.array_equal(G[s], G[s].T)


@pytest.mark.parametrize("N", [20, 50, 100])
def test_hessian_grad_soa_layout_is_the_same_numbers(mpc, N):
    """layout flag only permutes storage (the long-horizon kernel copies element-wise with 8-byte cp.async there)."""
    import torch
    import ntm_mpc
    from ntm_mpc import _lib
    S = 7
    rng = np.random.default_rng(N)
    Gam = rng.standard_normal((S, 2 * N, N)); Phi = rng.standard_normal((S, 2 * N, 2)); Lam = rng.standard_normal((S, 2 * N))
    X = sample_states(S, 3)
    phys, _, _ = o.make_batch(3, S=S)
    phys["q12"] = np.full(S, -0.2); phys["q22"] = np.full(S, 1.7)
    P = np.ascontiguousarray(o.derive_params_batch(phys).T)
    G0, F0 = mpc.hessian_grad(Phi, Gam, Lam, X, P)                                   # MATLAB layout
    dev = torch.device("cuda:0")
    soa = lambda a: torch.from_numpy(np.ascontiguousarray(a.reshape(S, -1).T)).to(dev)   # element index slowest
    # per-scenario blocks are column-major (MATLAB): Gamma(:,:,s) -> 2N*N elements in column-major order
    gam = soa(np.ascontiguousarray(Gam.transpose(0, 2, 1))); phi = soa(np.ascontiguousarray(Phi.transpose(0, 2, 1)))
    lam = soa(Lam); xx = soa(X); pp = soa(P)
    G = torch.empty(N * N * S, dtype=torch.float64, device=dev); F = torch.empty(N * S, dtype=torch.float64, device=dev)
    lib = _lib.load()
    mpc.set_stream(torch.cuda.current_stream(dev).cuda_stream or None)
    try:
        _lib.check(lib.ntm_hessian_grad_dev(mpc._h, ntm_mpc.LAYOUT_SOA, S, N, phi.data_ptr(), gam.data_ptr(), lam.data_ptr(),
                                            xx.data_ptr(), pp.data_ptr(), S, G.data_ptr(), F.data_ptr()))
        Gs = G.cpu().numpy().reshape(N * N, S).T.reshape(S, N, N); Fs = F.cpu().numpy().reshape(N, S).T
    finally:
        mpc.reset_stream()
    assert rel(Gs, G0) < 1e-12 and rel(Fs, F0) < 1e-12


# ------------------------------------------------------------------ getWLc.m (state-constraint condensation)
@pytest.mark.parametrize("N", [1, 3, 10, 20, 100])
def test_getWLc_matches_oracle_bit_for_bit(mpc, N):
    S = 5
    phys, _, _ = o.make_batch(3, S=S)
    R1, R2, R3 = _rho_batch(phys, S, N, 400 + N)
    Phi = np.zeros((S, 2 * N, 2)); Gam = np.zeros((S, 2 * N, N)); Lam = np.zeros((S, 2 * N))
    for s in range(S):
        Af, Bf, C = o.model_callables(o.scenario(phys, s))
        Phi[s], Gam[s], Lam[s] = o.Rho_to_PhiGammaLambda(R1[s], R2[s], R3[s], Af, Bf, C, s % 2)
    xmax, xmin, umax, umin = [0.15, 5000 * 2 * math.pi], [0.06, 100 * 2 * math.pi], [2e6], [0.0]       # NTM_MPC_Sim.m:40-50
    W, L, c = mpc.getWLc(xmax, xmin, umax, umin, Gam, Phi, Lam)
    assert W.shape == (S, 6 * N + 4, 2) and L.shape == (S, 6 * N + 4, N) and c.shape == (S, 6 * N + 4)
    for s in range(S):
        eW, eL, ec = o.getWLc(xmax, xmin, umax, umin, Gam[s], Phi[s], Lam[s])
        assert np.array_equal(W[s], eW) and np.array_equal(L[s], eL) and np.array_equal(c[s], ec)    # selection + sign only: exact
    # the rows mean what getWLc.m says: L U <= c + W x  <=>  umin <= U <= umax and xmin <= x_i <= xmax along the prediction
    U = np.random.default_rng(N).uniform(0, 2e6, N); x = np.array([0.1, 3000.0])
    X = np.concatenate([x, Phi[0] @ x + Gam[0] @ U + Lam[0]]).reshape(N + 1, 2)
    lhs = L[0] @ U - c[0] - W[0] @ x
    inside = np.all((X >= xmin) & (X <= xmax), axis=1)
    for i in range(N):
        assert bool(np.all(lhs[6 * i + 2:6 * i + 6] <= 1e-9 * np.abs(c[0][6 * i + 2:6 * i + 6]).max())) == bool(inside[i])
    assert np.all(lhs[0:6 * N:6] <= 0) and np.all(lhs[1:6 * N:6] <= 0)


# ------------------------------------------------------------------ box QP
def _random_qp(N, rng, cond_pow):
    M = rng.standard_normal((2 * N, N)) * np.logspace(0, -cond_pow / 2, N)[None, :]
    G = 2 * M.T @ M
    F = rng.standard_normal(N) * np.abs(G).max() * rng.uniform(0.1, 3)
    return G, F


@pytest.mark.parametrize("N", [1, 2, 3, 10, 20, 32, 33, 64, 100, 128])
def test_qp_box_kkt_and_oracle(mpc, N):
    rng = np.random.default_rng(300 + N)
    S = 24
    G = np.zeros((S, N, N)); F = np.zeros((S, N)); lb = np.zeros((S, N)); ub = np.zeros((S, N))
    for s in range(S):
        G[s], F[s] = _random_qp(N, rng, cond_pow=int(rng.integers(0, 7)))
        lb[s] = -rng.uniform(0.1, 2); ub[s] = rng.uniform(0.1, 2)
    U, it, st = mpc.qp_box(G, F, lb, ub)
    assert np.all(st == 0), st
    assert np.all(U >= lb) and np.all(U <= ub)
    for s in range(S):
        assert o.qp_kkt_residual(G[s], F[s], lb[s], ub[s], U[s]) < 1e-9
        Uo, _, so = co.qp_box(G[s], F[s], lb[s], ub[s])
        assert so == 0
        obj = lambda u: 0.5 * u @ G[s] @ u + F[s] @ u
        assert abs(obj(U[s]) - obj(Uo)) <= 1e-10 * (abs(obj(Uo)) + 1e-300)
        # bound components are bit-exact bounds
        at = (Uo == lb[s]) | (Uo == ub[s])
        assert np.array_equal(U[s][at], Uo[at])
    assert np.all(it >= 1) and np.all(it <= 10 * N + 20)


def test_qp_box_reference_conditioning(mpc):
    """The reference's own Hessians (cond 1e6..2e9, raw watts): G, F from the oracle closed loop trace."""
    for x0, N in (([0.0, 2000 * math.pi], 3), ([0.08, 2000 * math.pi], 10), ([0.1, 3000.0], 20)):
        tr = []
        o.closed_loop(o.default_physics(), x0, N=N, k_sim=3, i_sim=4, profile=o.LITERAL_FIXED, trace=tr)
        G = np.stack([t["G"] for t in tr]); F = np.stack([t["F"] for t in tr])
        U, it, st = mpc.qp_box(G, F, 0.0, 2e6)
        assert np.all(st == 0)
        for s in range(len(tr)):
            Uo, _, _ = o.qp_box(G[s], F[s], 0.0, 2e6)
            assert np.max(np.abs(U[s] - Uo)) <= TOL_TRAJ * 2e6
            assert o.qp_kkt_residual(G[s], F[s], 0.0, 2e6, U[s]) < 1e-9


def test_qp_box_edge_cases(mpc):
    U, it, st = mpc.qp_box(np.array([[2.0]]), np.array([-2.0]), 0.0, 5.0)
    assert U[0, 0] == pytest.approx(1.0) and st[0] == 0
    assert mpc.qp_box(np.array([[2.0]]), np.array([-2.0]), 2.0, 5.0)[0][0, 0] == 2.0
    assert mpc.qp_box(np.array([[2.0]]), np.array([-2.0]), -3.0, 0.5)[0][0, 0] == 0.5
    assert mpc.qp_box(np.array([[2.0]]), np.array([-2.0]), 0.25, 0.25)[0][0, 0] == 0.25      # degenerate box
    U, it, st = mpc.qp_box(np.array([[np.nan]]), np.array([-2.0]), 0.0, 1.0)
    assert st[0] == 2 and np.isnan(U[0, 0])
    G = np.array([[1.0, 2.0], [2.0, 1.0]])                                                    # indefinite: flagged, finite
    U, it, st = mpc.qp_box(G, np.array([-1.0, -1.0]), -10.0, 10.0)
    assert st[0] != 0 or o.qp_kkt_residual(G, np.array([-1.0, -1.0]), -10, 10, U[0]) < 1e-9


# ------------------------------------------------------------------ closed loop vs golden fixtures
@pytest.mark.parametrize("cfg", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("name", ["literal_fixed", "literal", "consistent_fixed"])
def test_closed_loop_matches_golden(mpc, cfg, name):
    g = np.load(os.path.join(GOLD, f"closed_loop_config{cfg}.npz"))
    if f"{name}_xk" not in g.files:
        pytest.skip("fixture not generated for this profile (N=100 oracle cost)")
    if cfg == 1 and name == "literal":
        pytest.skip("default scenario + 1e-14 stop rule is bit-chaotic by construction (SURVEY D14)")
    S, N = int(g["S"]), int(g["N"])
    r = mpc.closed_loop(g["x0"], g["params"].T, N=N, profile=int(g[f"{name}_flags"]), want_Uk=True)
    umax = g["phys_umax"]
    du, dw, dom = traj_err(r["uk"], r["xk"], g[f"{name}_uk"], g[f"{name}_xk"], umax)
    assert du.max() <= TOL_TRAJ and dw.max() <= TOL_TRAJ and dom.max() <= TOL_TRAJ, (du.max(), dw.max(), dom.max())
    assert np.max(np.abs(r["Uk"] - g[f"{name}_Uk"]) / umax[:, None, None]) <= TOL_TRAJ
    assert np.allclose(r["cost"], g[f"{name}_cost"], rtol=1e-6)
    assert np.all(r["status"] == 0)
    if name.endswith("fixed"):
        assert np.all(r["inner_iters"] == 10)
    else:
        assert np.mean(r["inner_iters"] == g[f"{name}_inner"]) >= 0.97


# ------------------------------------------------------------------ closed loop vs the C oracle, larger samples
@pytest.mark.parametrize("cfg,S", [(2, 1024), (3, 2048), (4, 2048), (5, 256)])
@pytest.mark.parametrize("prof", [o.LITERAL_FIXED, o.LITERAL], ids=["lit_fixed", "lit_eps"])
def test_closed_loop_matches_c_oracle_literal(mpc, cfg, S, prof):
    """Config 5 (N = 100, the sweep-tableau kernel of ntm_long.cuh) on 256 scenarios (round 1: 16)."""
    phys, x0, N = o.make_batch(cfg, S=S)
    P = o.derive_params_batch(phys)
    r = mpc.closed_loop(x0, P.T, N=N, profile=prof.flags())
    c = co.closed_loop_batch(phys, x0, N, flags=prof.flags())
    du, dw, dom = traj_err(r["uk"], r["xk"], c["uk"], c["xk"], phys["umax"])
    assert du.max() <= TOL_TRAJ and dw.max() <= TOL_TRAJ and dom.max() <= TOL_TRAJ, (du.max(), dw.max(), dom.max())
    assert np.allclose(r["cost"], c["cost"], rtol=1e-6)
    assert np.all(r["status"] == 0) and np.all(c["status"] == 0)
    assert np.mean(r["inner_iters"] == c["inner_iters"]) >= 0.99


@pytest.mark.parametrize("cfg,S", [(2, 1024), (3, 2048), (4, 2048)])
def test_closed_loop_consistent_profile_vs_c_oracle(mpc, cfg, S):
    """The 'consistent' reading is numerically touchier (SURVEY 0.5: an FMA-vs-no-FMA build of the *same* C
    oracle already disagrees on ~2e-4 of the scenarios at N=20), so parity is asserted on the quantile."""
    phys, x0, N = o.make_batch(cfg, S=S)
    P = o.derive_params_batch(phys)
    prof = o.CONSISTENT_FIXED
    r = mpc.closed_loop(x0, P.T, N=N, profile=prof.flags())
    c = co.closed_loop_batch(phys, x0, N, flags=prof.flags())
    du, dw, dom = traj_err(r["uk"], r["xk"], c["uk"], c["xk"], phys["umax"])
    ok = (du <= TOL_TRAJ) & (dw <= TOL_TRAJ) & (dom <= TOL_TRAJ)
    assert ok.mean() >= 0.995, ok.mean()
    assert np.median(du) <= 1e-9


def test_heaviest_scenarios_of_config3_alone(mpc):
    """Scenarios 62,420 / 60,466 / 60,091 of config 3 end the slowest 8-GPU shard (profiles/README.md: 10 bang-bang switches
    per QP, or ~10 free variables in every QP).  Parity with the C oracle on exactly these, and a guard on the QP start
    rule: from a previous solution scenario 62,420 needs 27 active-set iterations per QP (5,431 in all), from the best of
    four candidates 11 -- the sticky switch of qp_solve must have caught it."""
    idx = np.array([62420, 60466, 60091])
    phys, x0, N = o.make_batch(3, S=int(idx.max()) + 1)
    sub = {k: np.asarray(v)[idx].copy() for k, v in phys.items()}
    P = o.derive_params_batch(sub)
    prof = o.LITERAL_FIXED
    r = mpc.closed_loop(x0[idx], P.T, N=N, profile=prof.flags())
    c = co.closed_loop_batch(sub, x0[idx], N, flags=prof.flags())
    du, dw, dom = traj_err(r["uk"], r["xk"], c["uk"], c["xk"], sub["umax"])
    assert du.max() <= TOL_TRAJ and dw.max() <= TOL_TRAJ and dom.max() <= TOL_TRAJ, (du, dw, dom)
    assert np.all(r["status"] == 0)
    assert int(r["qp_iters"][0].sum()) <= 3000, r["qp_iters"].sum(axis=1)


def test_dense_and_toeplitz_hessian_paths_agree(mpc):
    import ntm_mpc
    P, x0, N = ntm_mpc.physics.batch_params(3, S=512)
    a = mpc.closed_loop(x0, P.T, N=N, profile=ntm_mpc.PROFILE_INNER_FIXED)
    b = mpc.closed_loop(x0, P.T, N=N, profile=ntm_mpc.PROFILE_INNER_FIXED | ntm_mpc.PROFILE_DENSE_G)
    du, dw, dom = traj_err(a["uk"], a["xk"], b["uk"], b["xk"], P[9])
    assert du.max() <= TOL_TRAJ and dw.max() <= TOL_TRAJ


@pytest.mark.parametrize("N,cfg", [(40, 3), (63, 3), (100, 5), (103, 5)])
def test_dense_hessian_on_the_tensor_cores_long_horizons(mpc, N, cfg):
    """Multi-warp dense-Gamma instantiation (build_GF_dense_dmma_long: Gamma streamed in 16-row chunks, Gamma' Omega Gamma
    by DMMA on 8 x 8 tiles, accumulators in registers): the literal reading forced through it (NTM_PROFILE_DENSE_G) gives
    the Toeplitz path's trajectories; N = 100 is BASELINE config 5's "dense contraction on FP64 tensor cores"."""
    import ntm_mpc
    phys, x0, _ = o.make_batch(cfg, S=48)
    P = o.derive_params_batch(phys)
    a = mpc.closed_loop(x0, P.T, N=N, k_sim=6, profile=ntm_mpc.PROFILE_INNER_FIXED)
    b = mpc.closed_loop(x0, P.T, N=N, k_sim=6, profile=ntm_mpc.PROFILE_INNER_FIXED | ntm_mpc.PROFILE_DENSE_G)
    du, dw, dom = traj_err(a["uk"], a["xk"], b["uk"], b["xk"], phys["umax"])
    assert np.all(b["status"] == 0)
    assert (du > TOL_TRAJ).sum() <= 1 and (dw > TOL_TRAJ).sum() <= 1, (N, float(du.max()), float(dw.max()))
    assert np.median(du) <= 1e-9


def test_closed_loop_variants_and_sizes(mpc):
    """rho1 'sq' variant, odd horizons across the warp/CTA group boundaries, k_sim/i_sim edge values."""
    phys, x0, _ = o.make_batch(3, S=8)
    P = o.derive_params_batch(phys)
    for N, flags in ((1, 0), (2, 16), (7, 1 | 16), (31, 16), (32, 16), (33, 16), (48, 16), (64, 16), (65, 16)):
        r = mpc.closed_loop(x0, P.T, N=N, k_sim=4, i_sim=3, profile=flags)
        c = co.closed_loop_batch(phys, x0, N, k_sim=4, i_sim=3, flags=flags)
        du, dw, dom = traj_err(r["uk"], r["xk"], c["uk"], c["xk"], phys["umax"])
        assert du.max() <= TOL_TRAJ and dw.max() <= TOL_TRAJ, (N, flags, du.max(), dw.max())
    # maximum horizon (NTM_MAX_HORIZON = 128): G + full LDL' workspace exceed shared memory -> small workspace + global slab
    r = mpc.closed_loop(x0[:3], P.T[:3], N=128, k_sim=2, i_sim=2, profile=16)
    c = co.closed_loop_batch({k: v[:3] for k, v in phys.items()}, x0[:3], 128, k_sim=2, i_sim=2, flags=16)
    du, dw, dom = traj_err(r["uk"], r["xk"], c["uk"], c["xk"], phys["umax"][:3])
    assert du.max() <= TOL_TRAJ and dw.max() <= TOL_TRAJ, (du.max(), dw.max())
    r = mpc.closed_loop(x0, P.T, N=5, k_sim=0, i_sim=1)
    assert np.array_equal(r["xk"][:, 0, :], x0)
    r = mpc.closed_loop(np.zeros((0, 2)), P.T[:0], N=5)                  # empty batch
    assert r["uk"].shape == (0, 20)


def test_nonfinite_scenarios_are_flagged_not_hidden(mpc):
    p = o.derive_params(o.default_physics())
    x0 = np.array([[0.08, 0.0], [0.08, 2000 * math.pi], [np.nan, 1.0]])      # omega = 0 -> rho2 = inf
    r = mpc.closed_loop(x0, p, N=5, k_sim=3, i_sim=2, profile=16)
    assert r["status"][0] == 2 and r["status"][2] == 2 and r["status"][1] == 0
    assert np.all(np.isfinite(r["xk"][1]))


# ------------------------------------------------------------------ randomised sweep
def test_randomised_sweep_of_horizons_profiles_and_loop_lengths(mpc):
    """60 random (N, S, k_sim, i_sim, profile bits) draws against the C oracle.  Literal readings (any rho1 variant, both
    inner policies, both Hessian builds) at the BASELINE horizons N <= 20 are held to 1e-6 on every trajectory.

    Longer horizons and the non-literal F / plant / Gamma-index readings contain scenarios on which NO fp64 implementation
    is within 1e-6 of the reference algorithm: adjudicated in 50-digit arithmetic (tools/adjudicate.py, table in
    profiles/r02_adjudication.txt) the NumPy oracle, the C oracle and the CUDA kernels each sit 1e-5 .. 1e-4 (sometimes a
    whole bang-bang switch) away from the exact closed loop and ~1e-6 .. 1e-4 away from each other -- an interior input
    of an ill-conditioned QP (cond 1e9+), not a kernel defect; on one of them the CUDA result is the only one within 1e-6.
    Measured rate (tools/find_chaotic.py, 2,048 scenarios per point, literal): 0 of 16,384 at N <= 24, 1-4 of 2,048
    (<= 0.2 %) at N = 32 .. 48.  Hence: a draw may lose ONE scenario, and the sweep at most 0.3 % of its scenarios."""
    rng = np.random.default_rng(4242)
    total_bad = total = 0
    for t in range(60):
        cfg = int(rng.choice([2, 3, 4]))
        N = int(rng.choice([1, 2, 3, 5, 8, 10, 13, 16, 20, 24, 31, 32, 33, 40, 48]))
        S = int(rng.integers(1, 120)); k_sim = int(rng.integers(1, 10)); i_sim = int(rng.integers(1, 11))
        flags = 0
        for bit, prob in ((1, 0.3), (2, 0.2), (4, 0.25), (8, 0.25), (16, 0.5)):
            if rng.random() < prob:
                flags |= bit
        if rng.random() < 0.15 and not flags & 2:
            flags |= 32
        phys, x0, _ = o.make_batch(cfg, S=S, seed=int(rng.integers(1, 1 << 30)))
        P = o.derive_params_batch(phys)
        g = mpc.closed_loop(x0, P.T, N=N, k_sim=k_sim, i_sim=i_sim, profile=flags)
        c = co.closed_loop_batch(phys, x0, N, k_sim=k_sim, i_sim=i_sim, flags=flags & 31)
        du, dw, dom = traj_err(g["uk"], g["xk"], c["uk"], c["xk"], phys["umax"])
        finite = np.isfinite(c["xk"]).all(axis=(1, 2)) & (c["status"] == 0)
        bad = ((du > TOL_TRAJ) | (dw > TOL_TRAJ)) & finite
        if flags & (2 | 4 | 8) or N > 20:
            assert bad.sum() <= 1, (t, N, S, flags, int(bad.sum()))
        else:
            assert not bad.any(), (t, N, S, flags, float(du.max()), float(dw.max()))
        total_bad += int(bad.sum()); total += S
        assert np.array_equal(np.isfinite(g["xk"]).all(axis=(1, 2)), np.isfinite(c["xk"]).all(axis=(1, 2)))
    print(f"randomised sweep: {total_bad} of {total} scenarios off by more than 1e-6")
    assert total_bad <= 0.003 * total, (total_bad, total)


# ------------------------------------------------------------------ full-size properties (BASELINE configs 3 / 4 shapes)
def test_full_size_properties_config3(mpc):
    import ntm_mpc
    P, x0, N = ntm_mpc.physics.batch_params(3)                               # 65,536 scenarios, N = 20
    S = x0.shape[0]
    prof = ntm_mpc.PROFILE_INNER_FIXED
    a = mpc.closed_loop(x0, P.T, N=N, profile=prof)
    b = mpc.closed_loop(x0, P.T, N=N, profile=prof)
    for k in ("xk", "uk", "cost", "inner_iters", "qp_iters", "status"):
        assert np.array_equal(a[k], b[k]), k                                 # run-to-run determinism (work queue order free)
    assert np.all(a["status"] == 0)
    assert np.all(a["uk"] >= P[8][:, None]) and np.all(a["uk"] <= P[9][:, None])   # box respected exactly
    # sharding invariance: any contiguous shard reproduces its slice bit-for-bit (scenarios are independent)
    for lo, hi in ((0, 8192), (8192, 8192 + 4099), (S - 5, S)):
        sh = mpc.closed_loop(x0[lo:hi], P.T[lo:hi], N=N, profile=prof)
        assert np.array_equal(sh["xk"], a["xk"][lo:hi]) and np.array_equal(sh["uk"], a["uk"][lo:hi])
    # closed-loop cost is what the trajectory says it is
    e = a["xk"][:, 1:, :] - np.stack([P[10], P[11]], axis=1)[:, None, :]
    cost = np.sum(P[12][:, None] * e[:, :, 0] ** 2 + 2 * P[13][:, None] * e[:, :, 0] * e[:, :, 1] + P[14][:, None] * e[:, :, 1] ** 2, axis=1)
    assert np.allclose(a["cost"], cost, rtol=1e-12)
    # a strided subsample agrees with the C oracle
    idx = np.arange(0, S, 97)
    phys, x0o, _ = o.make_batch(3)
    sub = {k: v[idx] for k, v in phys.items()}
    c = co.closed_loop_batch(sub, x0o[idx], N, flags=o.LITERAL_FIXED.flags())
    du, dw, dom = traj_err(a["uk"][idx], a["xk"][idx], c["uk"], c["xk"], sub["umax"])
    assert du.max() <= TOL_TRAJ and dw.max() <= TOL_TRAJ


def test_full_size_config4_bounds_active(mpc):
    import ntm_mpc
    P, x0, N = ntm_mpc.physics.batch_params(4, S=262144)                     # quarter of the 1,048,576 sweep per GPU
    r = mpc.closed_loop(x0, P.T, N=N, profile=0)
    assert np.all(r["status"] == 0)
    umax = P[9][:, None]
    at_ub = np.mean(r["uk"] == umax); at_lb = np.mean(r["uk"] == 0.0)
    assert at_ub > 0.01 and at_lb > 0.01 and at_ub + at_lb <= 1.0
    assert np.all((r["inner_iters"] >= 1) & (r["inner_iters"] <= 10))
    # a strided subsample of the full-size run agrees with the C oracle (round 1 only property-tested this size)
    idx = np.arange(0, 262144, 257)
    phys, x0o, _ = o.make_batch(4, S=262144)
    sub = {k: v[idx] for k, v in phys.items()}
    c = co.closed_loop_batch(sub, x0o[idx], N, flags=0)
    du, dw, dom = traj_err(r["uk"][idx], r["xk"][idx], c["uk"], c["xk"], sub["umax"])
    assert du.max() <= TOL_TRAJ and dw.max() <= TOL_TRAJ, (du.max(), dw.max())
    assert np.mean(r["inner_iters"][idx] == c["inner_iters"]) >= 0.99


def test_host_path_equals_resident_launch_on_a_large_batch(mpc):
    """Host-pointer entry (H2D, kernel, D2H inside the call) against the device-pointer entry on 16k+ scenarios, with and
    without the state rows: every output bit-identical.  (A chunked host path -- four launches, each chunk's D2H
    overlapping the next kernel -- passed this test but lost 19 % end to end: every launch pays the ~1 ms ramp-down of
    a persistent kernel whose scenarios take ~1 ms each; profiles/README.md.)"""
    import torch
    import ntm_mpc
    from ntm_mpc import physics
    S, N, ks = 16384 + 37, 5, 3
    P, x0, _ = physics.batch_params(3, S=S)
    prm = np.ascontiguousarray(P.T)
    for rows in (0, ntm_mpc.STATE_ROWS_REFRESH):
        xb = (0.05, 0.16, 2000.0, 12000.0)
        host = mpc.closed_loop(x0, prm, N=N, k_sim=ks, i_sim=4, profile=o.LITERAL_FIXED.flags(), want_Uk=True,
                               state_rows=rows, xbounds=xb if rows else None)
        dev = torch.device("cuda:0")
        dx = torch.from_numpy(x0).to(dev); dP = torch.from_numpy(prm).to(dev)
        xk = torch.empty((S, ks + 1, 2), dtype=torch.float64, device=dev); uk = torch.empty((S, ks), dtype=torch.float64, device=dev)
        Uk = torch.empty((S, ks, N), dtype=torch.float64, device=dev); cost = torch.empty(S, dtype=torch.float64, device=dev)
        inn = torch.empty((S, ks), dtype=torch.int32, device=dev); qp = torch.empty((S, ks), dtype=torch.int32, device=dev)
        st = torch.empty(S, dtype=torch.int32, device=dev)
        mpc.set_stream(torch.cuda.current_stream(dev).cuda_stream or None)
        try:
            args = (S, N, ks, 4, 1e-14, o.LITERAL_FIXED.flags(), ntm_mpc.LAYOUT_MATLAB, dx.data_ptr(), dP.data_ptr(), S)
            outs = (xk.data_ptr(), uk.data_ptr(), Uk.data_ptr(), cost.data_ptr(), inn.data_ptr(), qp.data_ptr(), st.data_ptr())
            if rows:
                mpc.closed_loop_sc_dev(*args, rows, xb, *outs)
            else:
                mpc.closed_loop_dev(*args, *outs)
            torch.cuda.synchronize()
        finally:
            mpc.reset_stream()
        for key, t in (("xk", xk), ("uk", uk), ("Uk", Uk), ("cost", cost), ("inner_iters", inn), ("qp_iters", qp), ("status", st)):
            assert np.array_equal(host[key], t.cpu().numpy(), equal_nan=True), (rows, key)


@pytest.mark.parametrize("N", [1, 3, 20, 40])
def test_getWLc_soa_layout_is_bit_identical(mpc, N):
    """SoA entry (one thread per scenario) against the MATLAB-layout path: a gather, so bit for bit."""
    import torch
    import ntm_mpc
    from ntm_mpc import _lib
    S = 41
    rng = np.random.default_rng(N + 7)
    Gam = rng.standard_normal((S, 2 * N, N)); Phi = rng.standard_normal((S, 2 * N, 2)); Lam = rng.standard_normal((S, 2 * N))
    xmax, xmin = [0.15, 3e4], [0.06, 600.0]
    W0, L0, c0 = mpc.getWLc(xmax, xmin, 2e6, 0.0, Gam, Phi, Lam)
    R = 6 * N + 4
    dev = torch.device("cuda:0")
    soa = lambda a: torch.from_numpy(np.ascontiguousarray(a.reshape(S, -1).T)).to(dev)
    gam = soa(np.ascontiguousarray(Gam.transpose(0, 2, 1))); phi = soa(np.ascontiguousarray(Phi.transpose(0, 2, 1))); lam = soa(Lam)
    W = torch.empty(R * 2 * S, dtype=torch.float64, device=dev); L = torch.empty(R * N * S, dtype=torch.float64, device=dev)
    c = torch.empty(R * S, dtype=torch.float64, device=dev)
    b = np.array([xmax[0], xmax[1], xmin[0], xmin[1], 2e6, 0.0])
    lib = _lib.load()
    mpc.set_stream(torch.cuda.current_stream(dev).cuda_stream or None)
    try:
        _lib.check(lib.ntm_getWLc_dev(mpc._h, ntm_mpc.LAYOUT_SOA, S, N, b.ctypes.data, gam.data_ptr(), phi.data_ptr(), lam.data_ptr(),
                                      W.data_ptr(), L.data_ptr(), c.data_ptr()))
        Ls = L.cpu().numpy().reshape(N, R, S).transpose(2, 1, 0); Ws = W.cpu().numpy().reshape(2, R, S).transpose(2, 1, 0)
        cs = c.cpu().numpy().reshape(R, S).T
    finally:
        mpc.reset_stream()
    assert np.array_equal(Ls, L0) and np.array_equal(Ws, W0) and np.array_equal(cs, c0)


# ------------------------------------------------------------------ layouts and error behaviour of the C ABI
def test_closed_loop_soa_layout_is_bit_identical_to_matlab_layout(mpc):
    import torch
    import ntm_mpc
    P, x0, N = ntm_mpc.physics.batch_params(4, S=777)
    S, ks = x0.shape[0], 6
    ref = mpc.closed_loop(x0, P.T, N=N, k_sim=ks, profile=0, want_Uk=True)
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    dx, dP = t(x0.T), t(P)                                               # SoA: element-major, scenario fastest
    xk = torch.empty((2 * (ks + 1), S), dtype=torch.float64, device=dev); uk = torch.empty((ks, S), dtype=torch.float64, device=dev)
    Uk = torch.empty((N * ks, S), dtype=torch.float64, device=dev); cost = torch.empty(S, dtype=torch.float64, device=dev)
    inner = torch.empty((ks, S), dtype=torch.int32, device=dev); qp = torch.empty((ks, S), dtype=torch.int32, device=dev)
    st = torch.empty(S, dtype=torch.int32, device=dev)
    mpc.set_stream(torch.cuda.current_stream().cuda_stream)
    mpc.closed_loop_dev(S, N, ks, 10, 1e-14, 0, ntm_mpc.LAYOUT_SOA, dx.data_ptr(), dP.data_ptr(), S, xk.data_ptr(), uk.data_ptr(),
                        Uk.data_ptr(), cost.data_ptr(), inner.data_ptr(), qp.data_ptr(), st.data_ptr())
    torch.cuda.synchronize()
    mpc.reset_stream()
    assert np.array_equal(xk.cpu().numpy().reshape(ks + 1, 2, S).transpose(2, 0, 1), ref["xk"])
    assert np.array_equal(uk.cpu().numpy().T, ref["uk"])
    assert np.array_equal(Uk.cpu().numpy().reshape(ks, N, S).transpose(2, 0, 1), ref["Uk"])
    assert np.array_equal(cost.cpu().numpy(), ref["cost"]) and np.array_equal(inner.cpu().numpy().T, ref["inner_iters"])
    assert np.array_equal(qp.cpu().numpy().T, ref["qp_iters"]) and np.array_equal(st.cpu().numpy(), ref["status"])


def test_c_abi_rejects_bad_arguments_with_a_message(mpc):
    import ctypes
    from ntm_mpc import _lib
    lib = _lib.load()
    h = mpc._h
    buf = np.zeros(4096)
    p = buf.ctypes.data
    ibuf = np.zeros(64, dtype=np.int32).ctypes.data
    def err():
        return lib.ntm_last_error().decode()
    assert lib.ntm_mpc_closed_loop(h, 0, 0, 1, 0, 20, 10, ctypes.c_double(1e-14), p, p, 1, p, p, None, p, ibuf, ibuf, ibuf) == 1 and "N out of range" in err()
    assert lib.ntm_mpc_closed_loop(h, 0, 0, 1, 129, 20, 10, ctypes.c_double(1e-14), p, p, 1, p, p, None, p, ibuf, ibuf, ibuf) == 1
    assert lib.ntm_mpc_closed_loop(h, 0, 0, 1, 3, 20, 0, ctypes.c_double(1e-14), p, p, 1, p, p, None, p, ibuf, ibuf, ibuf) == 1 and "i_sim" in err()
    assert lib.ntm_mpc_closed_loop(h, 7, 0, 1, 3, 20, 10, ctypes.c_double(1e-14), p, p, 1, p, p, None, p, ibuf, ibuf, ibuf) == 1 and "layout" in err()
    assert lib.ntm_mpc_closed_loop(h, 0, 0, 4, 3, 20, 10, ctypes.c_double(1e-14), p, p, 3, p, p, None, p, ibuf, ibuf, ibuf) == 1 and "params_count" in err()
    assert lib.ntm_mpc_closed_loop(h, 0, 0, 1, 3, 20, 10, ctypes.c_double(1e-14), None, p, 1, p, p, None, p, ibuf, ibuf, ibuf) == 1 and "NULL" in err()
    assert lib.ntm_rho(h, 0, 0, -1, p, p, 1, p, p, p) == 1 and "S must be" in err()
    assert lib.ntm_qp_box(h, 0, 2, 3, p, p, p, p, 5, p, ibuf, ibuf) == 1 and "bounds_count" in err()
    assert lib.ntm_condense(None, 0, 0, 1, 3, p, p, p, p, 1, p, p, p) == 1 and "handle" in err()
    # and the handle is still usable afterwards
    r1, _, _ = mpc.rho(np.array([[0.08, 6000.0]]), o.derive_params(o.default_physics()))
    assert np.isfinite(r1[0])


# ------------------------------------------------------------------ the reference's own names
def test_reference_named_api(mpc):
    import ntm_mpc as m
    p = o.default_physics()
    x = np.array([0.08, 2000 * math.pi])
    assert m.rho1(x, p["w_marg"]) == pytest.approx(o.rho1(x, p["w_marg"]), rel=1e-14)
    assert m.rho1(x, p["w_marg"], variant="sq") == pytest.approx(o.rho1(x, p["w_marg"], o.RHO1_SQ), rel=1e-14)
    assert m.rho2(x) == pytest.approx(o.rho2(x), rel=1e-14)
    assert m.rho3(x, p["w_dep"]) == pytest.approx(o.rho3(x, p["w_dep"]), rel=1e-14)
    kappa, zeta = o.kappa_of(p), o.zeta_of(p)
    args = (kappa, p["tau_r"], p["Ts"], zeta, p["rs"], p["a"], p["tau_E0"])
    Aref = o.A_mat(12.4, 1e-6, *args)
    assert rel(m.A(12.4, 1e-6, *args), Aref) < 1e-14
    assert rel(m.B(0.03, p["w_dep"], kappa, p["Ts"], p["eta_CD"]), o.B_mat(0.03, p["w_dep"], kappa, p["Ts"], p["eta_CD"])) < 1e-14
    # short call forms of the script resolve through the bound workspace (NTM_MPC_Sim.m:63-66,113)
    m.bind_workspace(m.workspace_from_physics(m.physics.nominal()))
    assert m.rho1(x) == m.rho1(x, p["w_marg"]) and m.rho3(x) == m.rho3(x, p["w_dep"])
    assert np.array_equal(m.A(12.4, 1e-6), m.A(12.4, 1e-6, *args))
    R = np.array([[12.0, 13.0, 14.0], [1e-6, 2e-6, 3e-6], [0.03, 0.04, 0.05]])
    Phi, Gam, Lam = m.Rho_to_PhiGammaLambda(R[0], R[1], R[2])
    Af, Bf, C = o.model_callables(p)
    e = o.Rho_to_PhiGammaLambda(R[0], R[1], R[2], Af, Bf, C)
    assert Phi.shape == (6, 2) and Gam.shape == (6, 3) and Lam.shape == (6,)
    assert rel(Phi, e[0]) < TOL_COND and rel(Gam, e[1]) < TOL_COND and rel(Lam, e[2]) < TOL_COND
    m.bind_workspace(None)
    with pytest.raises(TypeError):
        m.rho1(x)                                                           # "not enough input arguments"
    with pytest.raises(TypeError):
        m.Rho_to_PhiGammaLambda(R[0], R[1], R[2], lambda a, b: None, lambda a: None, C)
    G, F = o.hessian_grad(*e, x, [p["r1"], p["r2"]], np.eye(2))
    U, fval, flag = m.quadprog(G, F, lb=0.0, ub=2e6)
    assert flag == 1 and np.max(np.abs(U - o.qp_box(G, F, 0.0, 2e6)[0])) <= 1e-6 * 2e6
    xk, uk, Uk = m.NTM_MPC_Sim(inner_policy="fixed")
    ref = o.closed_loop(p, o.default_x0(), N=3, profile=o.LITERAL_FIXED)
    assert xk.shape == (2, 21) and uk.shape == (1, 20) and Uk.shape == (3, 20)
    assert np.max(np.abs(uk[0] - ref["uk"])) <= 1e-6 * 2e6
    assert np.max(np.abs(Uk - ref["Uk"])) <= 1e-6 * 2e6


def test_two_phase_longest_first_launch_is_bit_identical_to_the_single_launch():
    """Large one-warp box-loop batches run as two launches (time step 0, then the rest in longest-first order of a cost key
    from step 0, loop state carried through global memory): every output must equal the single launch in natural order bit
    for bit (tools/check_lpt.py, 16,384 scenarios, fixed / eps_break / config 4; NTM_LPT=0 is the single launch)."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "check_lpt.py"), "16384"], capture_output=True, text=True)
    assert r.returncode == 0 and "bit-identical: True" in r.stdout, r.stdout + r.stderr
