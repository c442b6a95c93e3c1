"""Replay of the box QPs the CUDA kernels solved, and a certificate for each answer (TEST INFRASTRUCTURE ONLY).

The closed loop is chaotic (DESIGN §2), so trajectory comparisons with the oracle carry allowances, and a wrong QP
answer can hide inside them.  Replaying removes the chaos: ``controller_step`` is stepped from the GPU's own measured
states with a ``qp`` callable that returns the U the GPU reported, so the oracle rebuilds every (G, F) the kernel
solved from the same x and the same previous U.  The argmin, the only non-smooth map of the loop, is replaced by the
GPU's answer; what is left between the two (G, F) is the rounding of the condensation.  Each GPU U is then certified
against its own QP (``certify``) and its partition compared with the oracle's where the oracle is unambiguous
(``partition_check``)."""
from __future__ import annotations

import copy
from typing import Callable, List, Sequence, Tuple

import numpy as np

from controller_oracle import controller_step
from oracle import ntm_oracle as o

# The kernels' own stop tests (csrc/ntm_long.cuh NTM_LONG_REFINE_TOL = 1e-9 on free components, csrc/ntm_device.cuh
# NTM_QP_EPS_G = 1e-13 on bound multipliers), with room for the rounding of the rebuilt (G, F) only.
FREE_TOL = 2e-9
MULT_TOL = 1e-11
# partition_check: a component is unambiguous when its oracle multiplier, or its distance to both bounds, exceeds this
AMBIGUOUS = 1e-6

QP = Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]      # (G, F, lb, ub)

# Profile flags (include/ntm_mpc.h) and the horizons at which the fused loop changes QP solver or workspace
# (launch_closed_loop, csrc/ntm_kernels.cu).  One warp (N <= 32): qp_solve<1>, whose LDL' workspace in shared memory is
# smaller than N from N = 22 (literal) / 16 (dense), larger free sets use the global slab.  Long literal: the sweep
# tableau in registers (33 <= N <= 104, 7 x 7 blocks) and in shared memory (105 <= N <= 128).  Multi-warp dense: the
# tensor-core build (N = 40, 103), the row sweep (N = 64, 104-128) and a 16-variable workspace from N = 116.
GAMMA_I, F_XK, FIXED, PLANT_RK4, DENSE_G = 2, 4, 16, 64, 32
ONE_WARP_LITERAL_N = (1, 12, 13, 20, 22, 24, 26, 31, 32)
ONE_WARP_DENSE_N = (16, 18, 26, 29, 32)
LONG_LITERAL_N = (33, 34, 41, 48, 63, 64, 65, 69, 97, 103, 104, 105, 111, 127, 128)
MULTI_WARP_DENSE_N = (40, 64, 103, 104, 116, 120, 128)


def profile_from_flags(flags: int) -> o.Profile:
    """The inverse of ``Profile.flags()``.  Bit 5 (``NTM_PROFILE_DENSE_G``, 32) is the dense build of the literal index:
    the same mathematics, so it maps to the literal profile."""
    if flags & 128:
        raise ValueError("TAUE_W: controller_step has no tau_E(w)")
    return o.Profile(rho1_variant=flags & 1, gamma_index=(flags >> 1) & 1, f_state=(flags >> 2) & 1,
                     plant_affine=(flags >> 3) & 1, inner_policy=(flags >> 4) & 1, plant_integrator=(flags >> 6) & 1)


class _Replay:
    """A ``qp`` for ``controller_step`` / ``closed_loop``: hands out the given solutions in order and records the QPs."""

    def __init__(self, Us: Sequence[np.ndarray]):
        self._Us = list(Us)
        self.qps: List[QP] = []

    def __call__(self, G, F, lb, ub):
        N = F.size
        self.qps.append((G.copy(), F.copy(), np.full(N, float(lb)), np.full(N, float(ub))))
        if len(self.qps) > len(self._Us):
            raise RuntimeError("the replay ran out of solutions")
        return np.array(self._Us[len(self.qps) - 1], dtype=np.float64), 0, 0


def replay_step(p, state: dict, x, Us: Sequence[np.ndarray], N: int, profile: o.Profile, eps: float = 1e-14) -> List[QP]:
    """One controller step at the measured state ``x`` whose inner QPs returned ``Us`` (in order).  ``state`` is the
    ``controller_step`` dict, advanced in place.  Returns the (G, F, lb, ub) of every QP of the step."""
    rp = _Replay(Us)
    controller_step(p, state, x, N, i_sim=len(Us), eps=eps, profile=profile, qp=rp)
    return rp.qps


def replay_fused(p, xk, Uk, N: int, profile: o.Profile) -> List[QP]:
    """The QPs of one scenario of a fused loop run with ``i_sim = 1``: ``xk`` [K+1, 2], ``Uk`` [K, N] as returned by
    ``closed_loop(..., i_sim=1, want_Uk=True)``.  With one inner iteration every QP the kernel solved is in ``Uk``."""
    state: dict = {}
    out: List[QP] = []
    for k in range(np.asarray(Uk).shape[0]):
        out += replay_step(p, state, xk[k], [Uk[k]], N, profile)
    return out


def prefix_solutions(step: Callable[[object, int], dict], record, I: int) -> List[dict]:
    """The results of one controller step cut after i = 1..I inner QPs: ``step(copy_of_record, i)``.  The controller is
    deterministic, so run i repeats the first i QPs of run I, and its U is the answer of QP i."""
    return [step(copy.deepcopy(record), i) for i in range(1, I + 1)]


def _scale(G, F, lb, ub):
    """s_j = |F_j| + sum_k |G_jk| max(|lb_k|, |ub_k|): the long solver's gradient scale (the rounding level of any
    gradient component inside the box).  Ratios against it are the same in U and in the literal kernels' y = b U."""
    return np.abs(F) + np.abs(G) @ np.maximum(np.abs(lb), np.abs(ub))


def _ratio(num, s):
    """num / s with 0 / 0 = 0 (a zero row of a semidefinite G with F_j = 0) and x / 0 = inf."""
    out = np.zeros_like(num)
    nz = s > 0
    out[nz] = num[nz] / s[nz]
    out[~nz & (num > 0)] = np.inf
    return out


def certify(G, F, lb, ub, U) -> dict:
    """KKT certificate of ``U`` for ``min 1/2 U'GU + F'U, lb <= U <= ub``, with g = GU + F in long double.  Returns the
    worst free-component ratio |g_j| / s_j, the worst bound-multiplier violation (-g_j / s_j at lb, g_j / s_j at ub,
    wrong sign only) and the worst infeasibility (max of lb - U, U - ub, inf for a non-finite U)."""
    ld = np.longdouble
    G = np.asarray(G, dtype=ld); F = np.asarray(F, dtype=ld).ravel(); U = np.asarray(U, dtype=np.float64).ravel()
    N = F.size
    lb = np.broadcast_to(np.asarray(lb, dtype=np.float64), (N,)); ub = np.broadcast_to(np.asarray(ub, dtype=np.float64), (N,))
    if not np.all(np.isfinite(U)):
        return dict(free=np.inf, mult=np.inf, infeas=np.inf)
    Ul = U.astype(ld)
    g = G @ Ul + F
    s = _scale(G, F, lb.astype(ld), ub.astype(ld))
    at_lb, at_ub = U == lb, U == ub
    free = (U > lb) & (U < ub)
    fr = _ratio(np.abs(g), s)
    mv = np.maximum(np.where(at_lb & ~at_ub, _ratio(-g, s), np.where(at_ub & ~at_lb, _ratio(g, s), 0)), 0)
    infeas = float(np.max(np.maximum(np.maximum(lb - U, U - ub), 0.0)))
    return dict(free=float(np.max(fr[free], initial=0.0)), mult=float(np.max(mv, initial=0.0)), infeas=infeas)


def passes(cert: dict) -> bool:
    return cert["free"] <= FREE_TOL and cert["mult"] <= MULT_TOL and cert["infeas"] == 0.0


def partition_check(G, F, lb, ub, U) -> Tuple[List[int], int]:
    """Compare the partition of ``U`` with ``o.qp_box`` on the same (G, F) where the oracle is unambiguous: an oracle
    bound component whose multiplier exceeds 1e-6 s_j must be that bound, bit for bit, and an oracle free component
    farther than 1e-6 of the width from both bounds must be free.  Returns (disagreeing components, skipped count);
    every component is skipped when the oracle does not reach a KKT point."""
    G = np.asarray(G, dtype=np.float64); F = np.asarray(F, dtype=np.float64).ravel(); U = np.asarray(U).ravel()
    N = F.size
    lb = np.broadcast_to(np.asarray(lb, dtype=np.float64), (N,)); ub = np.broadcast_to(np.asarray(ub, dtype=np.float64), (N,))
    Uo, _, st = o.qp_box(G, F, lb, ub)
    if st != 0:
        return [], N
    ld = np.longdouble
    g = np.asarray(G, dtype=ld) @ Uo.astype(ld) + np.asarray(F, dtype=ld)
    s = _scale(G.astype(ld), F.astype(ld), lb.astype(ld), ub.astype(ld))
    width = ub - lb
    bad, skipped = [], 0
    for j in range(N):
        if not width[j] > 0:
            skipped += 1
        elif Uo[j] == lb[j] and g[j] > AMBIGUOUS * s[j]:
            if U[j] != lb[j]:
                bad.append(j)
        elif Uo[j] == ub[j] and -g[j] > AMBIGUOUS * s[j]:
            if U[j] != ub[j]:
                bad.append(j)
        elif min(Uo[j] - lb[j], ub[j] - Uo[j]) > AMBIGUOUS * width[j]:
            if not lb[j] < U[j] < ub[j]:
                bad.append(j)
        else:
            skipped += 1
    return bad, skipped


def regime(phys: dict, x0: np.ndarray, name: str) -> dict:
    """A copy of a batch's physics with the QP-facing entries of the parameter block (umin, umax, r1, r2, q11, q12, q22:
    slots 8-14 of include/ntm_mpc.h) set for one regime:

    * ``natural``: unchanged;
    * ``wide``: umin = -umax, umax x 1e6 -- the minimisers are interior, so the free sets are the whole horizon;
    * ``wide10``: umin = -umax, umax x 10 -- mixed partitions;
    * ``reachable``: r1 = 0.8 w0, r2 = omega0 and q22 = 1e-9 (the omega error weighed like the w error), a reference
      the input can hold, so |U| is far below max(|lb|, |ub|) (the loosest scale);
    * ``pinned``: umin = umax; ``pinned_ulp``: umax = nextafter(umin);
    * ``semidefinite``: q11 = q12 = 0, so G = 2 Gamma' Omega Gamma only sees omega and is singular."""
    ph = {k: np.array(v, dtype=np.float64, copy=True) for k, v in phys.items()}
    S = x0.shape[0]
    umax = np.broadcast_to(ph["umax"], (S,)).copy()
    if name == "natural":
        pass
    elif name in ("wide", "wide10"):
        ph["umax"] = umax * (1e6 if name == "wide" else 10.0)
        ph["umin"] = -ph["umax"]
    elif name == "reachable":
        ph["r1"] = 0.8 * x0[:, 0]
        ph["r2"] = x0[:, 1].copy()
        ph["q22"] = np.full(S, 1e-9)
    elif name == "pinned":
        ph["umin"] = 0.5 * umax
        ph["umax"] = 0.5 * umax
    elif name == "pinned_ulp":
        ph["umin"] = 0.5 * umax
        ph["umax"] = np.nextafter(0.5 * umax, np.inf)
    elif name == "semidefinite":
        ph["q11"] = np.zeros(S)
        ph["q12"] = np.zeros(S)
    else:
        raise ValueError(name)
    return ph


class Worst:
    """Running worst certificate ratios and partition counts of a test case."""

    def __init__(self, name: str):
        self.name = name
        self.free = self.mult = self.infeas = 0.0
        self.nqp = self.skipped = self.ncomp = 0
        self.failures: List[str] = []

    def add(self, where, G, F, lb, ub, U, status_ok: bool = True, check_partition: bool = True):
        c = certify(G, F, lb, ub, U)
        self.nqp += 1
        self.ncomp += F.size
        self.free = max(self.free, c["free"]); self.mult = max(self.mult, c["mult"]); self.infeas = max(self.infeas, c["infeas"])
        if status_ok and not passes(c):
            self.failures.append(f"{where}: certificate {c}")
        if check_partition:
            bad, skipped = partition_check(G, F, lb, ub, U)
            self.skipped += skipped
            if bad:
                self.failures.append(f"{where}: partition differs from the oracle at {bad}")

    def report(self) -> str:
        return (f"[{self.name}] {self.nqp} QPs: worst free ratio {self.free:.2e}, multiplier violation {self.mult:.2e}, "
                f"infeasibility {self.infeas:.1e}, skipped {self.skipped} of {self.ncomp} components")
