"""The QP replay and certificate of tests/qp_replay.py, without a GPU.

Replaying the oracle's own closed loop rebuilds its (G, F) bit for bit, the certificate accepts exact solutions and
rejects answers that are wrong by 1e-7 of the box or on the wrong bound, and each regime of tests/test_gpu_loop_qp.py
produces on the oracle the QPs it claims (so the GPU file cannot quietly test nothing)."""
import copy
import dataclasses

import numpy as np
import pytest

import qp_replay as R
from controller_oracle import controller_step
from oracle import ntm_oracle as o

F_XK_ALONE = dataclasses.replace(o.LITERAL, f_state=o.F_XK)
GAMMA_I_ALONE = dataclasses.replace(o.LITERAL, gamma_index=o.GAMMA_I)
PROFILES = [("literal", o.LITERAL), ("consistent", o.CONSISTENT), ("f_xk", F_XK_ALONE), ("gamma_i", GAMMA_I_ALONE)]


def test_profile_from_flags_inverts_flags():
    for _, prof in PROFILES + [("fixed", o.LITERAL_FIXED), ("rk4", dataclasses.replace(o.CONSISTENT, plant_integrator=1))]:
        assert R.profile_from_flags(prof.flags()) == prof
    assert R.profile_from_flags(R.DENSE_G) == o.LITERAL
    assert R.profile_from_flags(R.DENSE_G | R.FIXED) == o.LITERAL_FIXED
    with pytest.raises(ValueError):
        R.profile_from_flags(128)


def offline_qp(p, x0, N, prof):
    Af, Bf, C = o.model_callables(p)
    r1 = o.rho1(x0, p["w_marg"], prof.rho1_variant)
    Phi, Gam, Lam = o.Rho_to_PhiGammaLambda(np.full(N, r1), np.full(N, o.rho2(x0)), np.full(N, o.rho3(x0, p["w_dep"])),
                                            Af, Bf, C, prof.gamma_index)
    return o.hessian_grad(Phi, Gam, Lam, x0, np.array([p["r1"], p["r2"]]),
                          np.array([[p["q11"], p["q12"]], [p["q12"], p["q22"]]]))


def assert_rebuilt(qps, trace, p, x0, N, prof):
    """QP n + 1 of the replay is solved on the (G, F) the oracle built after inner iteration n; QP 0 on the offline build."""
    assert len(qps) == len(trace)
    G0, F0 = offline_qp(p, x0, N, prof)
    assert np.array_equal(qps[0][0], G0) and np.array_equal(qps[0][1], F0)
    for n in range(len(trace) - 1):
        assert np.array_equal(qps[n + 1][0], trace[n]["G"]), n
        assert np.array_equal(qps[n + 1][1], trace[n]["F"]), n
    assert all(np.all(q[2] == p["umin"]) and np.all(q[3] == p["umax"]) for q in qps)


@pytest.mark.parametrize("N", [3, 20, 40])
@pytest.mark.parametrize("name,prof", PROFILES, ids=[c[0] for c in PROFILES])
def test_fused_replay_rebuilds_the_oracle_trace_bit_for_bit(name, prof, N):
    phys, x0, _ = o.make_batch(3, S=2)
    p = o.scenario(phys, 1)
    trace = []
    ref = o.closed_loop(p, x0[1], N=N, k_sim=6, i_sim=1, profile=prof, trace=trace)
    qps = R.replay_fused(p, ref["xk"].T, ref["Uk"].T, N, prof)
    assert_rebuilt(qps, trace, p, x0[1], N, prof)


@pytest.mark.parametrize("N", [3, 20, 40])
@pytest.mark.parametrize("prof", [o.LITERAL_FIXED, o.CONSISTENT_FIXED], ids=["literal_fixed", "consistent_fixed"])
def test_prefix_replay_rebuilds_every_inner_qp_bit_for_bit(prof, N):
    """The controller cut after i = 1..10 inner QPs gives the trace's U of QP i, and replaying those U through one
    10-iteration step rebuilds each (G, F)."""
    phys, x0, _ = o.make_batch(3, S=3)
    p = o.scenario(phys, 2)
    trace = []
    ref = o.closed_loop(p, x0[2], N=N, k_sim=3, i_sim=10, profile=prof, trace=trace)
    state, qps = {}, []
    for k in range(3):
        x = ref["xk"][:, k]
        pre = R.prefix_solutions(lambda st, i: controller_step(p, st, x, N, i_sim=i, profile=prof), state, 10)
        for i, r in enumerate(pre):
            assert np.array_equal(r["U"], trace[10 * k + i]["U"]), (k, i)
        keep = copy.deepcopy(state)
        qps += R.replay_step(p, state, x, [r["U"] for r in pre], N, prof)
        controller_step(p, keep, x, N, i_sim=10, profile=prof)
        for key in ("Rho1", "Rho2", "Rho3", "Uold", "G", "F"):
            assert np.array_equal(keep[key], state[key]), key
    assert_rebuilt(qps, trace, p, x0[2], N, prof)


# ------------------------------------------------------------------ the certificate
def oracle_qps(regime, N, S=4, K=4, prof=o.LITERAL, cfg=3):
    """(G, F, lb, ub, U_oracle) of the QPs of an oracle closed loop with i_sim = 1."""
    phys, x0, _ = o.make_batch(cfg, S=S)
    ph = R.regime(phys, x0, regime)
    out = []
    for s in range(S):
        p = o.scenario(ph, s)
        ref = o.closed_loop(p, x0[s], N=N, k_sim=K, i_sim=1, profile=prof)
        qps = R.replay_fused(p, ref["xk"].T, ref["Uk"].T, N, prof)
        out += [(*qp, U) for qp, U in zip(qps, ref["Uk"].T)]
    return out


@pytest.fixture(scope="module")
def mixed_qps():
    """Solved oracle QPs with free and bound components (config 3, umin = -umax, umax x 10, N = 20)."""
    out = []
    for G, F, lb, ub, _ in oracle_qps("wide10", 20):
        U, _, st = o.qp_box(G, F, lb, ub)
        free = (U > lb) & (U < ub)
        if st == 0 and free.any() and (~free).any():
            out.append((G, F, lb, ub, U))
    assert len(out) >= 4
    return out


def test_certify_accepts_exact_solutions(mixed_qps):
    for G, F, lb, ub, U in mixed_qps:
        c = R.certify(G, F, lb, ub, U)
        assert R.passes(c), c
        bad, skipped = R.partition_check(G, F, lb, ub, U)
        assert not bad and skipped < F.size


def _gradient(G, F, U):
    ld = np.longdouble
    return np.asarray(G, dtype=ld) @ U.astype(ld) + np.asarray(F, dtype=ld)


def test_certify_and_partition_check_reject_a_bound_flipped_to_the_other_bound(mixed_qps):
    for G, F, lb, ub, U in mixed_qps:
        g = _gradient(G, F, U)
        s = np.abs(F) + np.abs(G) @ np.maximum(np.abs(lb), np.abs(ub))
        lam = np.where(U == lb, g, np.where(U == ub, -g, -np.inf)).astype(np.float64) / s
        j = int(np.argmax(lam))                                         # the bound component the oracle is surest of
        assert lam[j] > R.AMBIGUOUS
        V = U.copy()
        V[j] = ub[j] if U[j] == lb[j] else lb[j]
        c = R.certify(G, F, lb, ub, V)
        assert not R.passes(c), c
        assert R.partition_check(G, F, lb, ub, V)[0] == [j]


def test_certify_rejects_a_free_component_nudged_by_1e_7_of_the_width(mixed_qps):
    for G, F, lb, ub, U in mixed_qps:
        free = np.flatnonzero((U > lb) & (U < ub))
        s = np.abs(F) + np.abs(G) @ np.maximum(np.abs(lb), np.abs(ub))
        j = int(free[np.argmax(np.diag(G)[free] * (ub - lb)[free] / s[free])])     # the component the nudge moves most
        V = U.copy()
        V[j] += 1e-7 * (ub[j] - lb[j]) * (1 if U[j] < 0.5 * (lb[j] + ub[j]) else -1)
        c = R.certify(G, F, lb, ub, V)
        assert c["free"] > R.FREE_TOL, c


def test_certify_rejects_a_bound_component_moved_1e_9_of_the_width_inside(mixed_qps):
    for G, F, lb, ub, U in mixed_qps:
        g = _gradient(G, F, U)
        lam = np.where(U == lb, g, np.where(U == ub, -g, -np.inf)).astype(np.float64)
        j = int(np.argmax(lam))
        assert lam[j] > 0
        V = U.copy()
        V[j] += 1e-9 * (ub[j] - lb[j]) * (1 if U[j] == lb[j] else -1)
        c = R.certify(G, F, lb, ub, V)
        assert c["free"] > R.FREE_TOL, c


def test_certify_rejects_infeasible_and_non_finite_answers(mixed_qps):
    G, F, lb, ub, U = mixed_qps[0]
    V = U.copy(); V[0] = np.nextafter(ub[0], np.inf)
    assert R.certify(G, F, lb, ub, V)["infeas"] > 0
    V[0] = np.nan
    assert not R.passes(R.certify(G, F, lb, ub, V))


def test_certify_handles_a_semidefinite_hessian_and_zero_data_without_0_over_0():
    qps = oracle_qps("semidefinite", 20, S=2, K=2)
    with np.errstate(all="raise"):
        for G, F, lb, ub, U in qps:
            N = F.size
            assert np.linalg.matrix_rank(G) < N                         # the last input reaches no predicted omega
            assert np.all(G[:, -1] == 0) and F[-1] == 0
            Uo, _, st = o.qp_box(G + np.diag(np.full(N, 1e-30)), F, lb, ub)   # any U_N is optimal
            c = R.certify(G, F, lb, ub, Uo)
            assert np.isfinite(c["free"]) and np.isfinite(c["mult"])
            assert c["mult"] <= R.MULT_TOL
        N = 5
        Z, lb, ub = np.zeros((N, N)), np.zeros(N), np.ones(N)
        for U in (np.zeros(N), np.ones(N), np.full(N, 0.3)):
            c = R.certify(Z, np.zeros(N), lb, ub, U)
            assert R.passes(c) and c == dict(free=0.0, mult=0.0, infeas=0.0)


# ------------------------------------------------------------------ the regimes of the GPU file, on the oracle
def free_sets(qps):
    return np.array([int(np.sum((U > lb) & (U < ub))) for _, _, lb, ub, U in qps])


# the horizons at which a free set can outgrow the one-warp shared-memory workspace or the 16-variable multi-warp one
SLAB = [(N, 0) for N in (22, 24, 26, 31, 32)] + [(N, R.GAMMA_I) for N in (16, 18, 26, 29, 32)] + \
       [(N, R.GAMMA_I) for N in (116, 120, 128)]


@pytest.mark.parametrize("N,flags", SLAB, ids=[f"N{N}_p{f}" for N, f in SLAB])
def test_wide_box_makes_the_whole_horizon_free(N, flags):
    qps = oracle_qps("wide", N, S=4 if N <= 32 else 2, K=4, prof=R.profile_from_flags(flags))
    fs = free_sets(qps)
    assert all(np.all(np.isfinite(U)) for *_, U in qps)
    assert np.median(fs) == N and fs.max() == N
    assert fs.max() > min(24, N - 1)                                     # above every one-warp workspace below N


def test_the_other_regimes_produce_what_they_claim():
    N = 20
    mixed = free_sets(oracle_qps("wide10", N))
    assert 0 < np.median(mixed) < N
    reach = oracle_qps("reachable", N)
    assert free_sets(reach).max() > 0
    assert np.median([np.max(np.abs(U)) / ub[0] for _, _, lb, ub, U in reach]) < 0.2
    for G, F, lb, ub, U in oracle_qps("pinned", N):
        assert np.all(lb == ub) and np.all(U == lb)
    for G, F, lb, ub, U in oracle_qps("pinned_ulp", N):
        assert np.all(ub == np.nextafter(lb, np.inf)) and np.all((U == lb) | (U == ub))
    for name in ("natural", "semidefinite"):
        assert all(np.all(np.isfinite(U)) for *_, U in oracle_qps(name, N))
