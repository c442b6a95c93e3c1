"""Per-call entry points of include/ntm_mpc.h (the ``*_dev`` twins) at batch sizes that wrap every launcher's grid or
persistent loop, in both layouts, on buffers that are 16-byte aligned or only 8 mod 16.

Every launcher caps its grid from the SM count and then loops over scenarios, so the code that only runs from a group's
second scenario on (prefetch of the next scenario, double-buffered staging, reused shared-memory tiles, the global LDL'
slab, accumulators that span scenarios) is only reached with S larger than one pass.  Four launchers also pick another
kernel or code path when a pointer is not 16-byte aligned.

Harness:
* ``pass_bound(family, N, sm)``: an upper bound on the scenarios one pass of a launch covers, from the SM count, the
  residency limits of sm_100 (64 warps and 32 CTAs per SM) and the launcher's own cap.  Wrapping sizes are
  ``S = 2 P + 37`` (every group at least two passes, some three), or ``P + 37`` where memory does not allow it.
* ``Buf``: each array sits inside a larger device buffer filled with a NaN sentinel of distinctive payload, with guard
  zones before and after it, at element offset 0 (16-byte aligned) or 1 (8 mod 16; asserted from the pointer).  After
  each call the guards must be unchanged, no output element may still hold the sentinel, and every input must be
  unchanged (two 64-bit fingerprints of its bits).
* Periodic inputs: scenario s gets input block ``s % M`` of M seeded blocks (M prime, not a divisor of the pass size,
  so the scenarios a group takes one after another differ).  A launch must then give every scenario the bits of its
  block's first scenario -- whatever the scheduler did -- and the references only need the M distinct blocks.
* Probes: the pass boundaries 0, 1, P-1, P, P+1, 2P-1, 2P, S-1 and 40 seeded indices, run again as a fresh, small,
  aligned batch that cannot wrap: same arithmetic, so the same bits.

Budget: about 3 minutes and 4 GB of device memory on one B200 (the lanes case of mc_stats is the largest, ~2.3 GB);
buffers are freed between cases.  Large inputs are generated on the device or tiled there from the M blocks; only the M
representatives travel to the host for the references.
"""
import math

import numpy as np
import pytest

import qp_replay as R
from oracle import ntm_oracle as o

MATLAB, SOA = 0, 1
LAYOUTS = ((MATLAB, "matlab"), (SOA, "soa"))
SM_MAX_WARPS, SM_MAX_CTAS = 64, 32            # residency limits of one sm_100 SM
GUARD = 64                                    # guard elements on each side of an array (512 bytes of doubles)
SENT64 = 0x7FF8_5EED_DEAD_BEEF                # quiet NaN, payload 0x85EEDDEADBEEF
SENT32 = 0x5EED_BEEF
WRAP_BYTES = 3 << 29                          # largest per-case working set for S = 2P + 37 (1.5 GB); beyond it P + 37
TOL_G, TOL_F = 1e-10, 1e-9                    # test_gpu_parity's tolerances of the Hessian entry
TOL_COND = 1e-10


# ------------------------------------------------------------------ pass sizes
def gw_for(N):
    return 1 if N <= 32 else (2 if N <= 64 else 4)       # csrc/ntm_kernels.cu gw_for


def resident(sm, warps_per_cta, groups_per_cta):
    """Most groups resident at once: CTAs per SM limited by 64 warps and 32 CTAs."""
    return sm * min(SM_MAX_WARPS // warps_per_cta, SM_MAX_CTAS) * groups_per_cta


def pass_bound(family, N, sm):
    """Upper bound on the scenarios one pass of the launch covers (csrc/ntm_kernels.cu)."""
    gw = gw_for(N)
    if family == "getwlc":            # launch_getwlc :236,240,244: min(S, 64 sm) CTAs, one scenario each
        return 64 * sm
    if family == "condense":          # launch_condense :1804-1808: 32 sm CTAs x 8 warps; :1819-1820: 16 sm CTAs
        return 32 * sm * 8 if N <= 32 else 16 * sm
    if family == "hessian_warp":      # launch_hessian_grad :1859-1867: persistent_geometry, 4 one-warp groups per CTA
        return resident(sm, 4, 4)
    if family == "hessian_dmma":      # :1838-1846: persistent_geometry, 256 threads, one scenario per CTA
        return resident(sm, 8, 1)
    if family == "hessian_generic":   # :1875-1889: hessian_grad_kernel<GW>, 32 GW threads, one scenario per CTA
        return resident(sm, gw, 1)
    if family == "qp_box":            # launch_qp_box :1670-1676: launch_persistent, group cap max_groups :1407
        wpb = 4 if gw == 1 else 1
        return min(resident(sm, gw * wpb, wpb), sm * (32 if gw == 1 else 4))
    if family == "qp_ineq":           # launch_qp_ineq :1688-1692: wpb <= 4 groups of GW warps, no group cap
        return sm * SM_MAX_WARPS // gw
    if family == "mc":                # launch_mc_stats :1710-1728: <= 64 warps per SM x 32 scenarios per warp pass
        return sm * SM_MAX_WARPS * 32
    raise ValueError(family)


def wrap_size(P, bytes_per_scenario, limit=WRAP_BYTES):
    S = 2 * P + 37
    return S if S * bytes_per_scenario <= limit else P + 37


def period(P, candidates=(97, 101, 103, 107, 109, 113)):
    return next(m for m in candidates if P % m)


def probes(S, P, seed, n=40):
    rng = np.random.default_rng(seed)
    edge = [0, 1, P - 1, P, P + 1, 2 * P - 1, 2 * P, S - 1]
    return np.unique(np.array([i for i in edge if 0 <= i < S] + list(rng.integers(0, S, n)), dtype=np.int64))


# ------------------------------------------------------------------ guarded device buffers
def _bits(t):
    import torch
    return t.view(torch.int64) if t.element_size() == 8 else t.view(torch.int32)


def fingerprint(t):
    """Two wrap-around 64-bit sums of the bits: plain, and weighted by position (catches moved elements)."""
    import torch
    v = _bits(t.reshape(-1)).to(torch.int64) if t.element_size() == 4 else _bits(t.reshape(-1))
    s1 = s2 = 0
    ch = 1 << 24
    for i in range(0, v.numel(), ch):
        c = v[i:i + ch]
        w = torch.arange(i, i + c.numel(), device=c.device, dtype=torch.int64) * 2 + 1
        s1 += int(c.sum()); s2 += int((c * w).sum())
    return s1 & (2 ** 64 - 1), s2 & (2 ** 64 - 1)


class Buf:
    """An array of n elements inside a larger device buffer whose guards and unwritten elements hold a sentinel.
    misalign: the array starts 8 bytes past a 16-byte boundary (doubles only)."""

    def __init__(self, n, dtype=None, misalign=False):
        import torch
        dtype = torch.float64 if dtype is None else dtype
        self.n, self.sent = int(n), (SENT64 if dtype == torch.float64 else SENT32)
        self.lo = GUARD + (1 if misalign else 0)
        self.base = torch.empty(self.lo + self.n + GUARD, dtype=dtype, device="cuda")
        _bits(self.base).fill_(self.sent)
        self.t = self.base[self.lo:self.lo + self.n]
        assert self.t.data_ptr() % 16 == (8 if misalign else 0), (self.t.data_ptr() % 16, misalign)
        self.fp = None                                   # set for inputs

    @property
    def ptr(self):
        return self.t.data_ptr()

    def fill(self, flat):
        self.t.copy_(flat.reshape(-1))
        self.fp = fingerprint(self.t)
        return self

    def check(self):
        lo, hi = _bits(self.base[:self.lo]), _bits(self.base[self.lo + self.n:])
        assert bool((lo == self.sent).all()) and bool((hi == self.sent).all()), "guard zone overwritten"
        if self.fp is None:
            assert not bool((_bits(self.t) == self.sent).any()), "output element left unwritten"
        else:
            assert fingerprint(self.t) == self.fp, "input modified"


def settle(*bufs):
    import torch
    torch.cuda.synchronize()
    for b in bufs:
        if b is not None:
            b.check()


def lay(blocks, layout):
    """[S, E] blocks -> the flat array of that layout."""
    return blocks.reshape(-1) if layout == MATLAB else blocks.t().contiguous().reshape(-1)


def blocks_of(t, S, layout):
    """flat array of a layout -> [S, E] view."""
    return t.view(S, -1) if layout == MATLAB else t.view(-1, S).t()


def put(src, sel, layout, misalign=False):
    """Input Buf holding src[sel % M] ([M, E] device blocks) in `layout`."""
    import torch
    d = src.index_select(0, torch.remainder(sel, src.shape[0]))
    return Buf(d.numel(), src.dtype, misalign).fill(lay(d, layout))


def out(S, E, misalign=False, dtype=None):
    return Buf(S * E, dtype, misalign)


def same_bits(a, b):
    return a.shape == b.shape and bool((_bits(a) == _bits(b)).all())


def assert_periodic(x, M):
    """x: [S, E] (any strides): every scenario carries the bits of scenario s % M."""
    import torch
    S = x.shape[0]
    ch = max(M, (1 << 22) // max(1, x.shape[1]) // M * M)
    for i in range(M, S, ch):
        c = x[i:min(S, i + ch)]
        rep = x.index_select(0, torch.arange(i, i + c.shape[0], device=x.device) % M)
        bad = (_bits(c) != _bits(rep)).any(dim=1)
        assert not bool(bad.any()), f"scenario {i + int(bad.nonzero()[0])} differs from its input's first scenario"


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-300))


# ------------------------------------------------------------------ fixtures
@pytest.fixture(scope="module")
def mpc():
    import torch
    import ntm_mpc
    h = ntm_mpc.NtmMpc(0)
    h.set_stream(torch.cuda.current_stream().cuda_stream)      # torch's stream: its copies and the kernels are ordered
    yield h
    h.reset_stream()
    h.close()


@pytest.fixture(scope="module")
def sm(mpc):
    return mpc.device_info()["sm_count"]


@pytest.fixture(autouse=True)
def _free_device_memory():
    yield
    import gc
    gc.collect()
    try:
        import torch
        if torch.cuda.is_available():
            torch.cuda.empty_cache()
    except ImportError:
        pass


def lib():
    from ntm_mpc import _lib
    return _lib.load()


def ok(rc):
    from ntm_mpc import _lib
    _lib.check(rc)


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda")


def sel_all(S):
    import torch
    return torch.arange(S, device="cuda")


# ------------------------------------------------------------------ references (each restates one oracle function)
def rho_blocks(M, N, seed):
    """Stage rho sequences from seeded states and the config-3 physics of M scenarios, and their parameter blocks."""
    rng = np.random.default_rng(seed)
    phys, _, _ = o.make_batch(3, S=M, seed=seed)
    P = np.ascontiguousarray(o.derive_params_batch(phys).T)               # [M, 16]
    w = rng.uniform(0.04, 0.16, (M, N)); om = rng.uniform(500.0, 14000.0, (M, N))
    R1 = o.rho1((w, om), phys["w_marg"][:, None]); R2 = o.rho2((w, om)); R3 = o.rho3((w, om), phys["w_dep"][:, None])
    return R1, R2, R3, P, phys


def condense_ref(R1, R2, R3, P, gamma_index):
    """Rho_to_PhiGammaLambda.m batched over the first axis, in np.longdouble.  Returns Phi [M, 2N, 2],
    Gamma [M, 2N, N], Lambda [M, 2N] (long double)."""
    ld = np.longdouble
    M, N = R1.shape
    P = P.astype(ld)
    a11 = P[:, 0:1] * R1.astype(ld) + 1                                    # A.m:2
    a21 = P[:, 1:2] * R2.astype(ld)
    b = P[:, 3:4] * R3.astype(ld)                                          # B.m:2
    a22, C1, C2 = P[:, 2], P[:, 4], P[:, 5]
    Phi = np.zeros((M, 2 * N, 2), dtype=ld); Gam = np.zeros((M, 2 * N, N), dtype=ld); Lam = np.zeros((M, 2 * N), dtype=ld)
    f11, f21, f22 = np.ones(M, dtype=ld), np.zeros(M, dtype=ld), np.ones(M, dtype=ld)
    l1, l2 = np.zeros(M, dtype=ld), np.zeros(M, dtype=ld)
    g1, g2 = np.zeros((M, N), dtype=ld), np.zeros((M, N), dtype=ld)
    for i in range(N):
        f11, f21, f22 = a11[:, i] * f11, a21[:, i] * f11 + a22 * f21, a22 * f22            # Phi_i = A_i Phi_{i-1}
        l1, l2 = a11[:, i] * l1 + C1, a21[:, i] * l1 + a22 * l2 + C2                        # Lambda_i = A_i Lambda_{i-1} + C
        Phi[:, 2 * i, 0], Phi[:, 2 * i + 1, 0], Phi[:, 2 * i + 1, 1] = f11, f21, f22
        Lam[:, 2 * i], Lam[:, 2 * i + 1] = l1, l2
        if i:                                                                               # blocks below the diagonal
            j = np.arange(i)
            k = np.full(i, i) if gamma_index else i - j - 1                                 # :32, A(Rho(i)) or A(Rho(i-j))
            n1 = a11[:, k] * g1[:, :i]
            n2 = a21[:, k] * g1[:, :i] + a22[:, None] * g2[:, :i]
            g1[:, :i], g2[:, :i] = n1, n2
        g1[:, i], g2[:, i] = b[:, i], 0                                                    # :36, B on the diagonal
        Gam[:, 2 * i, :i + 1], Gam[:, 2 * i + 1, :i + 1] = g1[:, :i + 1], g2[:, :i + 1]
    return Phi, Gam, Lam


def colmajor(a):
    """[M, rows, cols] -> [M, rows * cols] in MATLAB (column-major) block order."""
    return np.ascontiguousarray(np.asarray(a).transpose(0, 2, 1)).reshape(a.shape[0], -1)


def from_colmajor(flat, rows, cols):
    return np.asarray(flat).reshape(-1, cols, rows).transpose(0, 2, 1)


def getwlc_ref(Gam, Phi, Lam, bounds):
    """getWLc.m (D9 repaired) batched: a gather with signs, exact.  Zeros are +0.0 except c's -umin rows, as the kernels
    write them.  bounds = (xmax1, xmax2, xmin1, xmin2, umax, umin).  Returns W [M, R, 2], L [M, R, N], c [M, R]."""
    M, _, N = Gam.shape
    Rr = 6 * N + 4
    xmax, xmin, umax, umin = bounds[0:2], bounds[2:4], bounds[4], bounds[5]
    L = np.zeros((M, Rr, N)); W = np.zeros((M, Rr, 2)); c = np.zeros((M, Rr))
    for i in range(N + 1):
        r = 6 * i
        if i < N:
            L[:, r, i], L[:, r + 1, i] = -1.0, 1.0                                   # Ecal
            c[:, r], c[:, r + 1] = -umin, umax
            lo, hi = r + 2, r + 4
        else:
            lo, hi = r, r + 2                                                      # terminal rows MN, bN
        for comp in (0, 1):
            if i == 0:                                                             # block 0 constrains x_0: -Dcal
                W[:, lo + comp, comp], W[:, hi + comp, comp] = 1.0, -1.0
                c[:, lo + comp], c[:, hi + comp] = -xmin[comp], xmax[comp]
            else:
                row = 2 * (i - 1) + comp
                L[:, lo + comp], L[:, hi + comp] = -Gam[:, row], Gam[:, row]
                W[:, lo + comp], W[:, hi + comp] = Phi[:, row], -Phi[:, row]
                c[:, lo + comp], c[:, hi + comp] = -xmin[comp] + Lam[:, row], xmax[comp] - Lam[:, row]
    q0 = np.arange(0, 6 * N, 6)
    keep = c[:, q0].copy()
    L += 0.0; W += 0.0; c += 0.0                                                   # -0.0 -> +0.0
    c[:, q0] = keep
    return W, L, c


def mc_ref(xk, uk, cost, status, umin, umax, box, w_sup, hist_max, chunk=1 << 16):
    """o.mc_stats restated over device tensors (xk [S, K+1, 2], uk [S, K], cost, status, umin, umax [S], any strides):
    counts exact, sums per scenario on the device then math.fsum over scenarios."""
    import torch
    S, K = uk.shape
    outv = np.zeros(o.MC_NSTAT)
    outv[6] = outv[10] = np.inf; outv[7] = outv[11] = -np.inf
    parts = {i: [] for i in (4, 5, 8, 9, 18)}
    hist = torch.zeros(o.MC_NBINS, dtype=torch.int64, device=xk.device)
    cnt = np.zeros(o.MC_NSTAT, dtype=np.int64)
    for a in range(0, S, chunk):
        b = min(S, a + chunk)
        st = status[a:b].long()
        for k in range(4):
            cnt[k] += int((st == k).sum())
        idx = (st < 2).nonzero().squeeze(1) + a
        if idx.numel() == 0:
            continue
        x = xk.index_select(0, idx); u = uk.index_select(0, idx); cs = cost.index_select(0, idx)
        lo, hi = umin.index_select(0, idx), umax.index_select(0, idx)
        wf = x[:, K, 0]
        parts[4].append(cs); parts[5].append(cs * cs); parts[8].append(wf); parts[9].append(wf * wf)
        parts[18].append(u.sum(dim=1))
        outv[6] = min(outv[6], float(cs.min())); outv[7] = max(outv[7], float(cs.max()))
        outv[10] = min(outv[10], float(wf.min())); outv[11] = max(outv[11], float(wf.max()))
        cnt[12] += int((wf < w_sup).sum())
        below = x[:, 1:, 0] < w_sup
        reached = below.any(dim=1)
        first = torch.argmax(below.to(torch.int32), dim=1) + 1
        cnt[13] += int(first[reached].sum()); cnt[14] += int(reached.sum())
        cnt[15] += int((u <= lo[:, None]).sum()); cnt[16] += int((u >= hi[:, None]).sum()); cnt[17] += u.numel()
        w, om = x[:, 1:, 0], x[:, 1:, 1]
        cnt[19] += int(((w < box[0]) | (w > box[1])).sum()); cnt[20] += int(((om < box[2]) | (om > box[3])).sum())
        cnt[21] += w.numel()
        bins = torch.where(wf > 0, torch.floor(wf / hist_max * o.MC_NBINS), torch.zeros_like(wf)).long()
        hist += torch.bincount(bins.clamp(0, o.MC_NBINS - 1), minlength=o.MC_NBINS)
    for i, p in parts.items():
        outv[i] = math.fsum(torch.cat(p).cpu().numpy()) if p else 0.0
    for i in (0, 1, 2, 3, 12, 13, 14, 15, 16, 17, 19, 20, 21):
        outv[i] = cnt[i]
    outv[22:] = hist.cpu().numpy()
    return outv


MC_COUNTS = [0, 1, 2, 3, 12, 13, 14, 15, 16, 17, 19, 20, 21] + list(range(22, 22 + o.MC_NBINS))
MC_EXTREMA = [6, 7, 10, 11]
MC_SUMS = [4, 5, 8, 9, 18]
MC_BOX = (0.06, 0.15, 100 * 2 * np.pi, 5000 * 2 * np.pi)


def assert_mc_equal(got, exp):
    assert np.array_equal(got[MC_COUNTS], exp[MC_COUNTS]), (got[MC_COUNTS], exp[MC_COUNTS])
    assert np.array_equal(got[MC_EXTREMA], exp[MC_EXTREMA]), (got[MC_EXTREMA], exp[MC_EXTREMA])
    for i in MC_SUMS:
        assert abs(got[i] - exp[i]) <= 1e-12 * abs(exp[i]), (i, got[i], exp[i])


# ------------------------------------------------------------------ CPU: the references restate the oracle
def test_pass_bounds_wrap_and_probes_cover_the_boundaries():
    for sm in (132, 148, 160):
        for fam, N in (("getwlc", 20), ("condense", 32), ("condense", 100), ("hessian_warp", 7), ("hessian_dmma", 128),
                       ("hessian_generic", 20), ("qp_box", 10), ("qp_box", 128), ("qp_ineq", 20), ("mc", 20)):
            P = pass_bound(fam, N, sm)
            S = wrap_size(P, 8)
            assert S > 2 * P and P % period(P)
            p = probes(S, P, 1)
            assert {0, 1, P - 1, P, P + 1, 2 * P - 1, 2 * P, S - 1} <= set(p.tolist()) and p.max() < S
            assert len(p) <= sm                         # the probe batch never wraps a launch of one CTA per SM
    assert pass_bound("qp_box", 128, 148) == 4 * 148 and pass_bound("condense", 20, 148) == 256 * 148


@pytest.mark.parametrize("gi", [0, 1])
@pytest.mark.parametrize("N", [1, 2, 7, 20])
def test_condense_reference_is_the_oracle(N, gi):
    R1, R2, R3, P, phys = rho_blocks(5, N, 40 + N)
    Phi, Gam, Lam = condense_ref(R1, R2, R3, P, gi)
    for s in range(5):
        Af, Bf, C = o.model_callables(o.scenario(phys, s))
        eP, eG, eL = o.Rho_to_PhiGammaLambda(R1[s], R2[s], R3[s], Af, Bf, C, gi)
        assert rel(Phi[s], eP) < 1e-13 and rel(Gam[s], eG) < 1e-13 and rel(Lam[s], eL) < 1e-13
        assert np.array_equal(Gam[s] == 0, eG == 0) and np.array_equal(Phi[s] == 0, eP == 0)


@pytest.mark.parametrize("N", [1, 3, 10])
def test_getwlc_reference_is_the_oracle(N):
    rng = np.random.default_rng(N)
    Gam = rng.standard_normal((4, 2 * N, N)); Phi = rng.standard_normal((4, 2 * N, 2)); Lam = rng.standard_normal((4, 2 * N))
    b = (0.15, 3e4, 0.06, 600.0, 2e6, 0.0)
    W, L, c = getwlc_ref(Gam, Phi, Lam, b)
    for s in range(4):
        eW, eL, ec = o.getWLc(b[0:2], b[2:4], b[4], b[5], Gam[s], Phi[s], Lam[s])
        assert np.array_equal(W[s], eW) and np.array_equal(L[s], eL) and np.array_equal(c[s], ec)
    assert not np.any(np.signbit(L) & (L == 0)) and not np.any(np.signbit(W) & (W == 0))


def test_mc_reference_is_the_oracle():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(3)
    S, K = 500, 9
    xk, uk, cost, status, umax = _mc_host_batch(rng, S, K)
    exp = o.mc_stats(xk, uk, cost, status, 0.0, umax, MC_BOX, 0.06, 0.2)
    t = torch.from_numpy
    got = mc_ref(t(xk), t(uk), t(cost), t(status), t(np.zeros(S)), t(umax), MC_BOX, 0.06, 0.2, chunk=128)
    assert_mc_equal(got, exp)


def _mc_host_batch(rng, S, K):
    xk = rng.uniform(0.0, 0.2, (S, K + 1, 2)); xk[:, :, 1] = rng.uniform(0.0, 4e4, (S, K + 1))
    umax = rng.uniform(0.5e6, 2e6, S)
    uk = rng.uniform(0.0, 1.0, (S, K)) * umax[:, None]
    uk[rng.random((S, K)) < 0.3] = 0.0
    hit = rng.random((S, K)) < 0.3
    uk[hit] = np.broadcast_to(umax[:, None], (S, K))[hit]
    cost = rng.uniform(0.0, 10.0, S)
    status = rng.integers(0, 4, S).astype(np.int32)
    bad = status >= 2
    xk[bad, 1:, :] = np.nan; uk[bad] = np.nan; cost[bad] = np.nan
    return xk, uk, cost, status, umax


# ------------------------------------------------------------------ getWLc
WLC_BOUNDS = (0.15, 5000 * 2 * np.pi, 0.06, 100 * 2 * np.pi, 2e6, 0.0)      # xmax, xmin, umax, umin (NTM_MPC_Sim.m:40-50)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 3, 10, 20])
def test_getwlc_dev_wrapping_every_path_bit_for_bit(mpc, sm, N):
    """launch_getwlc (:237-244): getwlc_vec_kernel when all six pointers are 16-byte aligned, getwlc_kernel when any
    is not (Gamma only, c only, all six), getwlc_soa_kernel in SoA.  Every scenario equals the batched gather."""
    Rr = 6 * N + 4
    P = pass_bound("getwlc", N, sm)
    S = wrap_size(P, 8 * (Rr * (N + 3) + 2 * N * N + 6 * N))
    M = period(P)
    assert S > 2 * P
    rng = np.random.default_rng(500 + N)
    Gam = rng.standard_normal((M, 2 * N, N)); Phi = rng.standard_normal((M, 2 * N, 2)); Lam = rng.standard_normal((M, 2 * N))
    Gam[:, 1::2, :] *= 1e3                                                             # omega rows, other scale
    r, cidx = np.indices((2 * N, N))
    Gam[:, (r < 2 * cidx) | (r == 2 * cidx + 1)] = 0.0                                 # a condensed Gamma's exact zeros
    eW, eL, ec = getwlc_ref(Gam, Phi, Lam, WLC_BOUNDS)
    src = {k: dev(v) for k, v in (("gam", colmajor(Gam)), ("phi", colmajor(Phi)), ("lam", Lam))}
    b = np.array(WLC_BOUNDS)

    def run(sel, layout, mis=()):
        n = int(sel.numel())
        ins = {k: put(src[k], sel, layout, k in mis) for k in src}
        W, L, c = out(n, 2 * Rr, "W" in mis), out(n, N * Rr, "L" in mis), out(n, Rr, "c" in mis)
        ok(lib().ntm_getWLc_dev(mpc._h, layout, n, N, b.ctypes.data, ins["gam"].ptr, ins["phi"].ptr, ins["lam"].ptr,
                                W.ptr, L.ptr, c.ptr))
        settle(*ins.values(), W, L, c)
        return [blocks_of(x.t, n, layout) for x in (W, L, c)]

    ref = [dev(colmajor(eW)), dev(colmajor(eL)), dev(ec)]
    pr = dev(probes(S, P, N))
    alone = run(pr, MATLAB)
    for layout, mis in ((MATLAB, ()), (MATLAB, ("gam",)), (MATLAB, ("c",)), (MATLAB, ("gam", "phi", "lam", "W", "L", "c")),
                        (SOA, ())):
        got = run(sel_all(S), layout, mis)
        for g, r, a in zip(got, ref, alone):
            assert same_bits(g[:M], r), (layout, mis)
            assert_periodic(g, M)
            assert same_bits(g.index_select(0, pr), a), (layout, mis)
        del got


# ------------------------------------------------------------------ condense
@pytest.mark.gpu
@pytest.mark.parametrize("gi", [0, 1])
@pytest.mark.parametrize("N", [1, 20, 32, 33, 64, 100, 128])
def test_condense_dev_wrapping_both_layouts_and_alignments(mpc, sm, N, gi):
    """launch_condense (:1795-1822): condense_kernel<1> (N <= 32) / <2>, <4> with vec_ok (warp scan or staged index-i
    tiles, 16-byte stores) when Phi, Gamma, Lambda are 16-byte aligned, the generic per-element path when they are
    8 mod 16, condense_soa_kernel in SoA.  Every scenario within 1e-10 of the long-double recurrence."""
    P = pass_bound("condense", N, sm)
    E = 4 * N + 2 * N * N + 2 * N
    S = wrap_size(P, 8 * (E + 3 * N + 16))
    M = period(P)
    assert S > 2 * P
    R1, R2, R3, Pm, _ = rho_blocks(M, N, 600 + N)
    ePhi, eGam, eLam = condense_ref(R1, R2, R3, Pm, gi)
    eP, eG, eL = colmajor(ePhi).astype(np.float64), colmajor(eGam).astype(np.float64), eLam.astype(np.float64)
    src = {"r1": dev(R1), "r2": dev(R2), "r3": dev(R3), "p": dev(Pm)}
    flags = o.Profile(gamma_index=gi).flags()

    def run(sel, layout, mis=False, shared_params=None):
        n = int(sel.numel())
        ins = {k: put(src[k], sel, layout) for k in ("r1", "r2", "r3")}
        prm = Buf(16).fill(dev(shared_params)) if shared_params is not None else put(src["p"], sel, layout)
        Phi, Gam, Lam = out(n, 4 * N, mis), out(n, 2 * N * N, mis), out(n, 2 * N, mis)
        ok(lib().ntm_condense_dev(mpc._h, layout, flags, n, N, ins["r1"].ptr, ins["r2"].ptr, ins["r3"].ptr, prm.ptr,
                                  1 if shared_params is not None else n, Phi.ptr, Gam.ptr, Lam.ptr))
        settle(*ins.values(), prm, Phi, Gam, Lam)
        return [blocks_of(x.t, n, layout) for x in (Phi, Gam, Lam)]

    pr = dev(probes(S, P, N + gi))
    for layout, _ in LAYOUTS:
        alone = run(pr, layout)
        reps = {}
        for mis in (False, True):
            got = run(sel_all(S), layout, mis)
            for g, a in zip(got, alone):
                assert_periodic(g, M)
                if not mis:
                    assert same_bits(g.index_select(0, pr), a)
            reps[mis] = [g[:M].cpu().numpy() for g in got]
            del got
        for mis, (gP, gG, gL) in reps.items():
            for s in range(M):
                assert rel(gP[s], eP[s]) < TOL_COND and rel(gG[s], eG[s]) < TOL_COND and rel(gL[s], eL[s]) < TOL_COND, (layout, mis, s)
            assert np.array_equal(gG == 0, eG == 0) and np.array_equal(gP == 0, eP == 0)
        for a, u in zip(reps[False], reps[True]):                     # the two paths differ in arithmetic only
            assert rel(u, a) <= 1e-12 and np.array_equal(u == 0, a == 0)
    # params_count = 1 gives the bits of the replicated block
    for layout, _ in LAYOUTS:
        sel = sel_all(S)
        one = run(sel, layout, shared_params=Pm[0])
        src["p"] = dev(np.broadcast_to(Pm[0], (M, 16)))
        rep = run(sel, layout)
        src["p"] = dev(Pm)
        for a, b in zip(one, rep):
            assert same_bits(a, b)
        del one, rep


# ------------------------------------------------------------------ Hessian and gradient
def hessian_blocks(M, N, seed):
    rng = np.random.default_rng(seed)
    Gam = rng.standard_normal((M, 2 * N, N)); Phi = rng.standard_normal((M, 2 * N, 2)); Lam = rng.standard_normal((M, 2 * N))
    X = np.column_stack([rng.uniform(0.0, 0.2, M), rng.uniform(300.0, 30000.0, M)])
    phys, _, _ = o.make_batch(3, S=M, seed=seed)
    phys["q12"] = rng.uniform(-0.4, 0.4, M); phys["q22"] = rng.uniform(0.5, 3.0, M)
    Pm = np.ascontiguousarray(o.derive_params_batch(phys).T)
    ref = [o.hessian_grad(Phi[m], Gam[m], Lam[m], X[m], Pm[m, 10:12], np.array([[Pm[m, 12], Pm[m, 13]], [Pm[m, 13], Pm[m, 14]]]))
           for m in range(M)]
    return dict(gam=colmajor(Gam), phi=colmajor(Phi), lam=Lam, x=X, p=Pm), ref


HESS_SOA_GENERIC_N = (7, 20, 32)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 7, 8, 20, 31, 32, 33, 64, 100, 128])
def test_hessian_grad_dev_wrapping_every_path(mpc, sm, N):
    """launch_hessian_grad (:1835-1889).  N <= 32, MATLAB: hessian_grad_dmma_warp_kernel with aligned16 (16-byte copies
    and stores, even N) when Gamma and G are 16-byte aligned, 8-byte copies when Gamma or G is 8 mod 16 (double-
    buffered slices, padding rows re-zeroed per scenario at odd N).  N <= 32, SoA: hessian_grad_kernel<1>.  N > 32:
    hessian_grad_dmma_kernel in both layouts with vec16 (Gamma 16-byte aligned, MATLAB) or 8-byte copies, next-scenario
    prefetch of v.  Every launch: each scenario the bits of its input's first scenario and of the probe batch; the
    oracle at 1e-10 (G) / 1e-9 (F); G exactly symmetric."""
    if N <= 32:
        variants = [(MATLAB, ()), (MATLAB, ("gam",)), (MATLAB, ("G",))] + ([(SOA, ())] if N in HESS_SOA_GENERIC_N else [])
    else:
        variants = [(MATLAB, ()), (MATLAB, ("gam",)), (SOA, ()), (SOA, ("gam",))]
    blocks, ref = None, None
    for layout, mis in variants:
        fam = "hessian_dmma" if N > 32 else ("hessian_warp" if layout == MATLAB else "hessian_generic")
        P = pass_bound(fam, N, sm)
        S = wrap_size(P, 8 * (2 * N * N + 7 * N + 18 + N * N))
        M = period(P)
        assert S > 2 * P
        if blocks is None or blocks[0] != M:
            b, ref = hessian_blocks(M, N, 700 + N)
            blocks = (M, {k: dev(v) for k, v in b.items()})
        src = blocks[1]

        def run(sel, mis_=()):
            n = int(sel.numel())
            ins = {k: put(src[k], sel, layout, k in mis_) for k in src}
            G, F = out(n, N * N, "G" in mis_), out(n, N)
            ok(lib().ntm_hessian_grad_dev(mpc._h, layout, n, N, ins["phi"].ptr, ins["gam"].ptr, ins["lam"].ptr,
                                          ins["x"].ptr, ins["p"].ptr, n, G.ptr, F.ptr))
            settle(*ins.values(), G, F)
            return blocks_of(G.t, n, layout), blocks_of(F.t, n, layout)

        pr = dev(probes(S, P, N))
        aG, aF = run(pr)
        G, F = run(sel_all(S), mis)
        for g, a in ((G, aG), (F, aF)):
            assert_periodic(g, M)
            assert same_bits(g.index_select(0, pr), a), (layout, mis)
        Gh, Fh = G[:M].cpu().numpy().reshape(M, N, N), F[:M].cpu().numpy()
        for m in range(M):
            assert rel(Gh[m], ref[m][0]) < TOL_G and rel(Fh[m], ref[m][1]) < TOL_F, (layout, mis, m)
            assert np.array_equal(Gh[m], Gh[m].T)
        del G, F


# ------------------------------------------------------------------ box QP
def qp_blocks(M, N, seed):
    """SPD G of condition 1 .. 1e6 (test_gpu_parity's _random_qp), and four box regimes by block: random, wide
    (interior minimiser: every variable free), pinned (lb = ub), one ulp wide."""
    rng = np.random.default_rng(seed)
    G = np.zeros((M, N, N)); F = np.zeros((M, N)); lb = np.zeros((M, N)); ub = np.zeros((M, N))
    for m in range(M):
        A = rng.standard_normal((2 * N, N)) * np.logspace(0, -int(rng.integers(0, 7)) / 2, N)[None, :]
        G[m] = 2 * A.T @ A
        G[m] = 0.5 * (G[m] + G[m].T)
        F[m] = rng.standard_normal(N) * np.abs(G[m]).max() * rng.uniform(0.1, 3)
        kind = m % 4
        if kind == 0:
            lb[m], ub[m] = -rng.uniform(0.1, 2, N), rng.uniform(0.1, 2, N)
        elif kind == 1:
            lb[m], ub[m] = -1e6, 1e6
        elif kind == 2:
            lb[m] = ub[m] = rng.uniform(-1, 1, N)
        else:
            lb[m] = rng.uniform(-1, 1, N); ub[m] = np.nextafter(lb[m], np.inf)
    return G, F, lb, ub


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 10, 32, 33, 64, 100, 128])
def test_qp_box_dev_wrapping_both_layouts(mpc, sm, N):
    """launch_qp_box (:1665-1676): qp_box_kernel<GW> pulls scenarios from the work queue; at N = 128 the LDL' workspace
    does not fit shared memory (hcap_qp :1401-1405) and the wide boxes' free sets run in the group's global slab.
    bounds_count S and 1, iters / status NULL once.  SoA = MATLAB bit for bit, every clean scenario certified."""
    import torch
    P = pass_bound("qp_box", N, sm)
    S = wrap_size(P, 8 * (2 * N * N + 5 * N))
    M = period(P)
    assert S > 2 * P
    G, F, lb, ub = qp_blocks(M, N, 800 + N)
    src = {"G": dev(G.transpose(0, 2, 1).reshape(M, -1)), "F": dev(F), "lb": dev(lb), "ub": dev(ub)}
    shared = (dev(np.full(N, -1.0)), dev(np.full(N, 1.0)))

    def run(sel, layout, bc, with_iters=True):
        n = int(sel.numel())
        ins = {k: put(src[k], sel, layout) for k in ("G", "F")}
        if bc == 1:
            ins["lb"], ins["ub"] = Buf(N).fill(shared[0]), Buf(N).fill(shared[1])
        else:
            ins["lb"], ins["ub"] = put(src["lb"], sel, layout), put(src["ub"], sel, layout)
        U = out(n, N)
        it, st = (out(n, 1, dtype=torch.int32), out(n, 1, dtype=torch.int32)) if with_iters else (None, None)
        ok(lib().ntm_qp_box_dev(mpc._h, layout, n, N, ins["G"].ptr, ins["F"].ptr, ins["lb"].ptr, ins["ub"].ptr,
                                1 if bc == 1 else n, U.ptr, it.ptr if it else None, st.ptr if st else None))
        settle(*ins.values(), U, it, st)
        return [blocks_of(U.t, n, layout)] + ([it.t.view(n, 1), st.t.view(n, 1)] if with_iters else [])

    pr = dev(probes(S, P, N))
    for bc in ("S", 1):
        res = {}
        for layout, name in LAYOUTS:
            res[name] = run(sel_all(S), layout, bc)
            alone = run(pr, layout, bc)
            for g, a in zip(res[name], alone):
                assert_periodic(g, M)
                assert same_bits(g.index_select(0, pr), a), (name, bc)
        for a, b in zip(res["matlab"], res["soa"]):
            assert same_bits(a, b), bc
        U, it, st = (x[:M].cpu().numpy() for x in res["matlab"])
        assert np.all(st == 0), (bc, st.ravel())
        assert np.all(it >= 0) and np.all(it <= 10 * N + 20)
        for m in range(M):
            lo, hi = (lb[m], ub[m]) if bc == "S" else (-1.0, 1.0)
            c = R.certify(G[m], F[m], lo, hi, U[m])
            assert R.passes(c), (bc, m, c)
        if bc == 1:
            Un = run(sel_all(S), MATLAB, bc, with_iters=False)[0]
            assert same_bits(Un, res["matlab"][0])
        del res


# ------------------------------------------------------------------ QP with getWLc's state rows
def ineq_blocks(M, N, seed):
    """First QP of a closed-loop step with getWLc's rows (test_gpu_qp_ineq._mpc_problems), split as the quadprog
    gateway does; every third problem gets one general row that no U in the box can meet (infeasible)."""
    rng = np.random.default_rng(seed)
    phys, x0, _ = o.make_batch(3, S=4 * M, seed=seed)
    out_ = []
    for s in range(4 * M):
        if len(out_) == M:
            break
        p = o.scenario(phys, s); x = x0[s].copy()
        Af, Bf, C = o.model_callables(p)
        xs = [x * (1 + 0.06 * rng.standard_normal(2)) for _ in range(N)]
        R1 = np.array([o.rho1(v, p["w_marg"]) for v in xs]); R2 = np.array([o.rho2(v) for v in xs])
        R3 = np.array([o.rho3(v, p["w_dep"]) for v in xs])
        Phi, Gam, Lam = o.Rho_to_PhiGammaLambda(R1, R2, R3, Af, Bf, C)
        Gm, Fm = o.hessian_grad(Phi, Gam, Lam, x, np.array([0.0, 2000 * np.pi]), np.eye(2))
        xmin = np.array([0.06, 100 * 2 * np.pi]); xmax = np.array([0.15, 5000 * 2 * np.pi])
        if s % 2:
            xmin[0] = x[0] * 0.9
        W, L, c = o.getWLc(xmax, xmin, 2e6, 0.0, Gam, Phi, Lam)
        lb, ub, Lg, bg, feas = o.split_rows(L, c + W @ x)
        if not (feas and np.all(np.isfinite(lb)) and np.all(np.isfinite(ub)) and np.all(lb < ub)):
            continue                                     # decided on the host side: never reaches the kernel
        if len(out_) % 3 == 2 and Lg.shape[0]:
            r = int(rng.integers(0, Lg.shape[0]))
            low = np.sum(np.minimum(Lg[r] * lb, Lg[r] * ub))
            bg = bg.copy(); bg[r] = low - 1e-2 * np.sum(np.abs(Lg[r]) * (ub - lb)) - 1e-3
        out_.append((Gm, Fm, lb, ub, Lg, bg))
    assert len({q[4].shape[0] for q in out_}) == 1
    return out_


@pytest.mark.gpu
@pytest.mark.parametrize("N", [3, 10, 20])
def test_qp_ineq_dev_wrapping_both_layouts(mpc, sm, N):
    """launch_qp_ineq (:1680-1693): qp_ineq_kernel<1> on the work queue.  SoA = MATLAB bit for bit; the oracle
    comparison of test_gpu_qp_ineq.py; status 3 exactly where the oracle finds the rows infeasible."""
    import torch
    P = pass_bound("qp_ineq", N, sm)
    M = 29 if P % 29 else 31                                            # the oracle's active set is slow: few blocks
    probs = ineq_blocks(M, N, 900 + N)
    Mr = probs[0][4].shape[0]
    S = wrap_size(P, 8 * (N * N + Mr * N + Mr + 4 * N))
    assert S > 2 * P and Mr > 0
    src = {"G": dev(np.stack([q[0].T.reshape(-1) for q in probs])), "F": dev(np.stack([q[1] for q in probs])),
           "lb": dev(np.stack([q[2] for q in probs])), "ub": dev(np.stack([q[3] for q in probs])),
           "Lg": dev(np.stack([q[4].T.reshape(-1) for q in probs])), "bg": dev(np.stack([q[5] for q in probs]))}

    def run(sel, layout):
        n = int(sel.numel())
        ins = {k: put(src[k], sel, layout) for k in src}
        U, it, st = out(n, N), out(n, 1, dtype=torch.int32), out(n, 1, dtype=torch.int32)
        ok(lib().ntm_qp_ineq_dev(mpc._h, layout, n, N, Mr, ins["G"].ptr, ins["F"].ptr, ins["lb"].ptr, ins["ub"].ptr, n,
                                 ins["Lg"].ptr, ins["bg"].ptr, U.ptr, it.ptr, st.ptr))
        settle(*ins.values(), U, it, st)
        return [blocks_of(U.t, n, layout), it.t.view(n, 1), st.t.view(n, 1)]

    pr = dev(probes(S, P, N))
    res = {}
    for layout, name in LAYOUTS:
        res[name] = run(sel_all(S), layout)
        alone = run(pr, layout)
        for g, a in zip(res[name], alone):
            assert_periodic(g, M)
            assert same_bits(g.index_select(0, pr), a), name
    for a, b in zip(res["matlab"], res["soa"]):
        assert same_bits(a, b)
    U, _, st = (x[:M].cpu().numpy() for x in res["matlab"])
    n_inf = 0
    for m, (Gm, Fm, lb, ub, Lg, bg) in enumerate(probs):
        Uo, _, so = o.qp_ineq(Gm, Fm, lb, ub, Lg, bg)
        assert st[m, 0] == so, (m, st[m, 0], so)
        if so == o.QP_INFEASIBLE:
            n_inf += 1
            continue
        assert np.max(np.abs(U[m] - Uo) / (ub - lb)) < 1e-6, m
        stat, viol = o.qp_ineq_kkt_residual(Gm, Fm, lb, ub, Lg, bg, U[m])
        assert stat < 1e-7 and viol < 1e-8, (m, stat, viol)
    assert 0 < n_inf < M


# ------------------------------------------------------------------ Monte-Carlo reduction
def mc_lanes_k(smem_optin):
    """Smallest k_sim whose staged tile exceeds the launcher's shared-memory budget (launch_mc_stats :1708-1710)."""
    K = 1
    while 32 * ((2 * (K + 1) | 1) + (K | 1)) * 8 <= smem_optin - 2048:
        K += 1
    return K


def mc_device_batch(S, K, seed, xk=None, uk=None):
    """Synthetic closed-loop results on the device (every status code; non-finite trajectories where status >= 2),
    written into xk [S, K+1, 2] and uk [S, K] when given (views of guarded buffers: no second copy of the largest case)."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    u = lambda *shape: torch.rand(*shape, generator=g, device="cuda", dtype=torch.float64)
    xk = torch.empty((S, K + 1, 2), dtype=torch.float64, device="cuda") if xk is None else xk
    uk = torch.empty((S, K), dtype=torch.float64, device="cuda") if uk is None else uk
    xk[:, :, 0] = u(S, K + 1) * 0.2
    xk[:, :, 1] = u(S, K + 1) * 4e4
    umax = 0.5e6 + 1.5e6 * u(S)
    uk.copy_(u(S, K) * umax[:, None])
    uk.masked_fill_(u(S, K) < 0.3, 0.0)
    hit = u(S, K) < 0.3
    uk[hit] = umax[:, None].expand(S, K)[hit]
    cost = 10.0 * u(S)
    status = torch.randint(0, 4, (S,), generator=g, device="cuda", dtype=torch.int32)
    bad = status >= 2
    xk[bad, 1:, :] = float("nan"); uk[bad] = float("nan"); cost[bad] = float("nan")
    return xk, uk, cost, status, umax


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["staged", "lanes", "soa"])
def test_mc_stats_dev_wrapping(mpc, sm, kind):
    """launch_mc_stats: mc_stats_matlab_kernel (staged tiles, k_sim = 20; also with xk / uk at 8 mod 16),
    mc_stats_matlab_lanes_kernel (the smallest k_sim above the staged kernel's shared-memory budget), mc_stats_soa_kernel.
    Through ntm_mc_stats_dev (parameter block) and ntm_mc_stats_ub_dev (compact umin / umax, bounds_count S and 1)."""
    import torch
    K = 20 if kind != "lanes" else mc_lanes_k(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)
    layout = SOA if kind == "soa" else MATLAB
    P = pass_bound("mc", 0, sm)
    S = wrap_size(P, 8 * (3 * K + 6 + 16), limit=2 << 30)
    assert S > P + 36 and (S > 2 * P or kind == "lanes")
    box = np.array(MC_BOX)
    exp1 = None
    for mis in ((False, True) if kind == "staged" else (False,)):
        bx, bu = Buf(S * (K + 1) * 2, misalign=mis), Buf(S * K, misalign=mis)
        if layout == MATLAB:
            xk, uk, cost, status, umax = mc_device_batch(S, K, 17 + K, bx.t.view(S, K + 1, 2), bu.t.view(S, K))
            bx.fp, bu.fp = fingerprint(bx.t), fingerprint(bu.t)
        else:
            xk, uk, cost, status, umax = mc_device_batch(S, K, 17 + K)
            bx.fill(lay(xk.view(S, -1), layout)); bu.fill(lay(uk, layout))
        assert set(status.unique().tolist()) == {0, 1, 2, 3}
        umin = torch.zeros(S, dtype=torch.float64, device="cuda")
        umin[::7] = 1e3                                                                 # a few nonzero lower bounds
        exp = mc_ref(xk, uk, cost, status, umin, umax, MC_BOX, 0.06, 0.2)
        bc = Buf(S).fill(cost); bs = Buf(S, dtype=torch.int32).fill(status)
        prm = torch.zeros((S, 16), dtype=torch.float64, device="cuda"); prm[:, 8] = umin; prm[:, 9] = umax
        bp = Buf(16 * S).fill(lay(prm, layout)); del prm
        bmin, bmax = Buf(S).fill(umin), Buf(S).fill(umax)
        o1, o2 = Buf(o.MC_NSTAT), Buf(o.MC_NSTAT)
        ok(lib().ntm_mc_stats_dev(mpc._h, layout, S, K, bx.ptr, bu.ptr, bc.ptr, bs.ptr, bp.ptr, S, box.ctypes.data,
                                  0.06, 0.2, o1.ptr))
        ok(lib().ntm_mc_stats_ub_dev(mpc._h, layout, S, K, bx.ptr, bu.ptr, bc.ptr, bs.ptr, bmin.ptr, bmax.ptr, S,
                                     box.ctypes.data, 0.06, 0.2, o2.ptr))
        settle(bx, bu, bc, bs, bp, bmin, bmax, o1, o2)
        assert_mc_equal(o1.t.cpu().numpy(), exp)
        assert_mc_equal(o2.t.cpu().numpy(), exp)
        if not mis:                                                                     # one shared pair
            if exp1 is None:
                exp1 = mc_ref(xk, uk, cost, status, torch.full_like(umin, 1e3), torch.full_like(umax, 1.5e6), MC_BOX, 0.06, 0.2)
            one = Buf(1).fill(torch.tensor([1e3], dtype=torch.float64, device="cuda"))
            two = Buf(1).fill(torch.tensor([1.5e6], dtype=torch.float64, device="cuda"))
            ok(lib().ntm_mc_stats_ub_dev(mpc._h, layout, S, K, bx.ptr, bu.ptr, bc.ptr, bs.ptr, one.ptr, two.ptr, 1,
                                         box.ctypes.data, 0.06, 0.2, o2.ptr))
            settle(bx, bu, one, two, o2)
            assert_mc_equal(o2.t.cpu().numpy(), exp1)
        del bx, bu, bp


# ------------------------------------------------------------------ rho, A/B, plant step
@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["rho", "lpv_AB", "plant_step"])
def test_elementwise_dev_layouts_alignment_and_shared_params(mpc, entry):
    """One thread per scenario, S not a multiple of 256: SoA = MATLAB bit for bit, also with every pointer 8 mod 16;
    params_count = 1 gives the bits of the replicated block."""
    S = 256 * 41 + 37
    rng = np.random.default_rng(len(entry))
    phys, _, _ = o.make_batch(3, S=S, seed=5)
    Pm = np.ascontiguousarray(o.derive_params_batch(phys).T)
    X = np.column_stack([rng.uniform(0.0, 0.2, S), rng.uniform(300.0, 30000.0, S)])
    ins = {"rho": {"x": X}, "lpv_AB": {"r1": rng.uniform(5, 300, (S, 1)), "r2": rng.uniform(0, 1e-4, (S, 1)),
                                       "r3": rng.uniform(0.01, 0.4, (S, 1))},
           "plant_step": {"x": X, "u": rng.uniform(0, 2e6, (S, 1))}}[entry]
    outs = {"rho": (1, 1, 1), "lpv_AB": (4, 2), "plant_step": (2,)}[entry]
    flags = o.Profile(plant_affine=1).flags()

    def run(layout, mis, params):
        pc = params.shape[0] if params.shape[0] == S else 1
        bi = {k: Buf(v.size, misalign=mis).fill(lay(dev(v.reshape(S, -1)), layout)) for k, v in ins.items()}
        bp = Buf(params.size, misalign=mis).fill(lay(dev(params), layout) if pc == S else dev(params))
        bo = [out(S, e, mis) for e in outs]
        h, L = mpc._h, lib()
        if entry == "rho":
            ok(L.ntm_rho_dev(h, layout, 0, S, bi["x"].ptr, bp.ptr, pc, *(b.ptr for b in bo)))
        elif entry == "lpv_AB":
            ok(L.ntm_lpv_AB_dev(h, layout, S, bi["r1"].ptr, bi["r2"].ptr, bi["r3"].ptr, bp.ptr, pc, *(b.ptr for b in bo)))
        else:
            ok(L.ntm_plant_step_dev(h, layout, flags, S, bi["x"].ptr, bi["u"].ptr, bp.ptr, pc, bo[0].ptr))
        settle(*bi.values(), bp, *bo)
        return [blocks_of(b.t, S, layout) for b in bo]

    base = run(MATLAB, False, Pm)
    for layout, mis in ((SOA, False), (MATLAB, True), (SOA, True)):
        for a, b in zip(base, run(layout, mis, Pm)):
            assert same_bits(a, b), (layout, mis)
    for layout, mis in ((MATLAB, False), (SOA, True)):
        one = run(layout, mis, Pm[7:8].reshape(1, 16))
        rep = run(layout, mis, np.ascontiguousarray(np.broadcast_to(Pm[7], (S, 16))))
        for a, b in zip(one, rep):
            assert same_bits(a, b), (layout, mis)


# ------------------------------------------------------------------ poison containment
POISON = (np.nan, np.inf, -np.inf)


def poison_rows(S, P, seed):
    """Every 5th scenario and every pass-boundary probe."""
    return np.unique(np.concatenate([np.arange(0, S, 5), probes(S, P, seed, n=0)]))


def plant(buf, S, layout, rows, cols):
    """Write NaN / +-Inf into the given element columns of the given scenarios of an input Buf (before freezing it)."""
    x = blocks_of(buf.t, S, layout)
    r = dev(rows)
    for i, cidx in enumerate(cols):
        x[r, cidx] = float(POISON[i % 3])
    buf.fp = fingerprint(buf.t)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["condense20", "condense20_gi", "condense100", "hessian7", "hessian20", "hessian64",
                                  "hessian100", "qp_box10", "qp_box64", "qp_box128", "qp_ineq10", "mc_stats"])
def test_poison_stays_in_its_scenario(mpc, sm, case):
    """NaN and +-Inf planted in every 5th scenario and every pass-boundary probe (rho entries for condense, Gamma for the
    Hessian, G or F for the QPs, xk with status 2 for mc_stats): every other scenario is bit-identical to the poison-free
    run, a poisoned QP comes back with status 2, and the reduction excludes the poisoned trajectories.  Padding is
    zero-filled and shared memory is never read stale, so 0 * NaN cannot carry a scenario into the next one."""
    import torch
    if case == "mc_stats":
        K, layout = 20, MATLAB
        P = pass_bound("mc", 0, sm)
        S = 2 * P + 37
        xk, uk, cost, status, umax = mc_device_batch(S, K, 99)
        rows = dev(poison_rows(S, P, 3))
        status[rows] = 2
        umin = torch.zeros(S, dtype=torch.float64, device="cuda")
        exp = mc_ref(xk, uk, cost, status, umin, umax, MC_BOX, 0.06, 0.2)
        xk[rows, 1:, 0] = float("nan"); xk[rows, :1, 1] = float("inf")
        box = np.array(MC_BOX)
        bx = Buf(xk.numel()).fill(xk); bu = Buf(uk.numel()).fill(uk); bc = Buf(S).fill(cost)
        bs = Buf(S, dtype=torch.int32).fill(status); bmin, bmax = Buf(S).fill(umin), Buf(S).fill(umax)
        o2 = Buf(o.MC_NSTAT)
        ok(lib().ntm_mc_stats_ub_dev(mpc._h, layout, S, K, bx.ptr, bu.ptr, bc.ptr, bs.ptr, bmin.ptr, bmax.ptr, S,
                                     box.ctypes.data, 0.06, 0.2, o2.ptr))
        settle(bx, bu, bc, bs, bmin, bmax, o2)
        assert_mc_equal(o2.t.cpu().numpy(), exp)
        return
    fam, N = {"condense20": ("condense", 20), "condense20_gi": ("condense", 20), "condense100": ("condense", 100),
              "hessian7": ("hessian", 7), "hessian20": ("hessian", 20), "hessian64": ("hessian", 64),
              "hessian100": ("hessian", 100), "qp_box10": ("qp_box", 10), "qp_box64": ("qp_box", 64),
              "qp_box128": ("qp_box", 128), "qp_ineq10": ("qp_ineq", 10)}[case]
    layout = MATLAB
    if fam == "hessian":
        P = pass_bound("hessian_dmma" if N > 32 else "hessian_warp", N, sm)
    else:
        P = pass_bound(fam, N, sm)
    S = 2 * P + 37
    M = period(P)
    rows = poison_rows(S, P, 3)
    rng = np.random.default_rng(N)
    if fam == "condense":
        R1, R2, R3, Pm, _ = rho_blocks(M, N, 1000 + N)
        src = {"r1": dev(R1), "r2": dev(R2), "r3": dev(R3), "p": dev(Pm)}
        names, poisoned, nout = ("r1", "r2", "r3", "p"), {"r1": [0, N - 1], "r2": [N // 2], "r3": [N - 1]}, (4 * N, 2 * N * N, 2 * N)

        def call(b, o_):
            ok(lib().ntm_condense_dev(mpc._h, layout, 2 if case.endswith("gi") else 0, S, N, b["r1"].ptr, b["r2"].ptr,
                                      b["r3"].ptr, b["p"].ptr, S, *(x.ptr for x in o_)))
    elif fam == "hessian":
        blk, _ = hessian_blocks(M, N, 1000 + N)
        src = {k: dev(v) for k, v in blk.items()}
        names, nout = ("phi", "gam", "lam", "x", "p"), (N * N, N)
        poisoned = {"gam": [0, 2 * N - 1, 2 * N * N - 1, int(rng.integers(0, 2 * N * N))]}

        def call(b, o_):
            ok(lib().ntm_hessian_grad_dev(mpc._h, layout, S, N, b["phi"].ptr, b["gam"].ptr, b["lam"].ptr, b["x"].ptr,
                                          b["p"].ptr, S, *(x.ptr for x in o_)))
    elif fam == "qp_box":
        G, F, lb, ub = qp_blocks(M, N, 1000 + N)
        src = {"G": dev(G.reshape(M, -1)), "F": dev(F), "lb": dev(lb), "ub": dev(ub)}
        names, nout = ("G", "F", "lb", "ub"), (N, 1, 1)
        poisoned = {"G": [0, N * N - 1], "F": [N // 2]}

        def call(b, o_):
            ok(lib().ntm_qp_box_dev(mpc._h, layout, S, N, b["G"].ptr, b["F"].ptr, b["lb"].ptr, b["ub"].ptr, S,
                                    *(x.ptr for x in o_)))
    else:
        probs = ineq_blocks(29 if P % 29 else 31, N, 1000 + N)
        M = len(probs)
        Mr = probs[0][4].shape[0]
        src = {"G": dev(np.stack([q[0].T.reshape(-1) for q in probs])), "F": dev(np.stack([q[1] for q in probs])),
               "lb": dev(np.stack([q[2] for q in probs])), "ub": dev(np.stack([q[3] for q in probs])),
               "Lg": dev(np.stack([q[4].T.reshape(-1) for q in probs])), "bg": dev(np.stack([q[5] for q in probs]))}
        names, nout = ("G", "F", "lb", "ub", "Lg", "bg"), (N, 1, 1)
        poisoned = {"G": [N + 1], "F": [0, N - 1]}

        def call(b, o_):
            ok(lib().ntm_qp_ineq_dev(mpc._h, layout, S, N, Mr, b["G"].ptr, b["F"].ptr, b["lb"].ptr, b["ub"].ptr, S,
                                     b["Lg"].ptr, b["bg"].ptr, *(x.ptr for x in o_)))
    is_qp = fam in ("qp_box", "qp_ineq")

    def run(poison):
        b = {k: put(src[k], sel_all(S), layout) for k in names}
        if poison:
            for k, cols in poisoned.items():
                plant(b[k], S, layout, rows, cols)
        o_ = [out(S, e, dtype=torch.int32 if (is_qp and i) else None) for i, e in enumerate(nout)]
        call(b, o_)
        settle(*b.values(), *o_)
        return [blocks_of(x.t, S, layout) for x in o_]

    clean, dirty = run(False), run(True)
    keep = torch.ones(S, dtype=torch.bool, device="cuda")
    keep[dev(rows)] = False
    for c, d in zip(clean, dirty):
        assert same_bits(c[keep], d[keep]), case
    if is_qp:
        assert bool((dirty[2][~keep] == 2).all()), dirty[2][~keep].unique()


# ------------------------------------------------------------------ one work queue, four launches, no host sync
@pytest.mark.gpu
def test_work_queue_rearm_under_load(mpc, sm):
    """qp_box_dev, qp_ineq_dev, qp_box_dev (another GW) and closed_loop_dev share the handle's work-queue counter; each
    launch's last group re-arms it (:293-297, :354-358).  Queued back to back on one stream with no host synchronisation,
    every result equals the same call run alone, bit for bit."""
    import torch
    from ntm_mpc import physics
    calls = []
    for N in (10, 33):
        P = pass_bound("qp_box", N, sm); S = 2 * P + 37; M = period(P)
        G, F, lb, ub = qp_blocks(M, N, 1100 + N)
        src = [dev(G.reshape(M, -1)), dev(F), dev(lb), dev(ub)]
        b = [put(t, sel_all(S), MATLAB) for t in src]
        o_ = [out(S, N), out(S, 1, dtype=torch.int32), out(S, 1, dtype=torch.int32)]
        calls.append((lambda b=b, o_=o_, S=S, N=N: ok(lib().ntm_qp_box_dev(mpc._h, MATLAB, S, N, *(x.ptr for x in b), S,
                                                                         *(x.ptr for x in o_))), b, o_))
    N = 10
    P = pass_bound("qp_ineq", N, sm); S = 2 * P + 37
    probs = ineq_blocks(29 if P % 29 else 31, N, 1200)
    Mr = probs[0][4].shape[0]
    src = [dev(np.stack([q[0].T.reshape(-1) for q in probs])), dev(np.stack([q[1] for q in probs])),
           dev(np.stack([q[2] for q in probs])), dev(np.stack([q[3] for q in probs])),
           dev(np.stack([q[4].T.reshape(-1) for q in probs])), dev(np.stack([q[5] for q in probs]))]
    b = [put(t, sel_all(S), MATLAB) for t in src]
    o_ = [out(S, N), out(S, 1, dtype=torch.int32), out(S, 1, dtype=torch.int32)]
    calls.insert(1, (lambda b=b, o_=o_, S=S: ok(lib().ntm_qp_ineq_dev(mpc._h, MATLAB, S, N, Mr, *(x.ptr for x in b[:4]), S,
                                                                      b[4].ptr, b[5].ptr, *(x.ptr for x in o_))), b, o_))
    Pm, x0, Nl = physics.batch_params(3, S=8192 + 37)
    S, ks = x0.shape[0], 4
    b = [Buf(x0.size).fill(dev(x0)), Buf(Pm.size).fill(dev(np.ascontiguousarray(Pm.T)))]
    o_ = [out(S, 2 * (ks + 1)), out(S, ks), out(S, Nl * ks), out(S, 1), out(S, ks, dtype=torch.int32),
          out(S, ks, dtype=torch.int32), out(S, 1, dtype=torch.int32)]
    calls.append((lambda b=b, o_=o_, S=S: mpc.closed_loop_dev(S, Nl, ks, 10, 1e-14, 16, MATLAB, b[0].ptr, b[1].ptr, S,
                                                              *(x.ptr for x in o_)), b, o_))
    alone = []
    for fn, b, o_ in calls:
        fn()
        settle(*b, *o_)
        alone.append([x.t.clone() for x in o_])
    for _, _, o_ in calls:
        for x in o_:
            _bits(x.t).fill_(x.sent)
    for fn, _, _ in calls:
        fn()
    for (_, b, o_), ref in zip(calls, alone):
        settle(*b, *o_)
        for x, r in zip(o_, ref):
            assert same_bits(x.t, r)
