"""Batched host API over the C ABI (include/ntm_mpc.h).  NumPy arrays in, NumPy arrays out; every
call runs the sm_100a kernels -- nothing here computes on the CPU.

Array convention ("MATLAB layout"): the leading axis is the scenario; the per-scenario block is the
MATLAB matrix in column-major order.  To keep NumPy indexing natural the returned arrays are views
shaped ``[S, rows, cols]`` (Fortran order inside each scenario block), e.g. ``Gamma[s]`` is the
2N x N matrix the reference's ``Rho_to_PhiGammaLambda`` would return for scenario ``s``.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional

import numpy as np

from . import _lib
from ._lib import LAYOUT_MATLAB, LAYOUT_SOA, NPARAM, NtmError, check, ctrl_doubles, load, rec_doubles  # noqa: F401

MC_NBINS = 32                                   # NTM_MC_NBINS / NTM_MC_NSTAT of include/ntm_mpc.h
MC_NSTAT = 22 + MC_NBINS
MC_STATE_BOX = (0.06, 0.15, 100 * 2 * 3.141592653589793, 5000 * 2 * 3.141592653589793)   # xmin(1), xmax(1), xmin(2), xmax(2): NTM_MPC_Sim.m:39-45


def _f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data


def _blocks_in(a, S: int, rows: int, cols: int) -> np.ndarray:
    """[S, rows, cols] (or [rows, cols] when S == 1) -> flat MATLAB layout."""
    a = np.asarray(a, dtype=np.float64)
    if a.ndim == 2:
        a = a[None]
    if a.shape != (S, rows, cols):
        raise ValueError(f"expected shape {(S, rows, cols)}, got {a.shape}")
    return np.ascontiguousarray(a.transpose(0, 2, 1))


def _blocks_out(flat: np.ndarray, S: int, rows: int, cols: int) -> np.ndarray:
    return flat.reshape(S, cols, rows).transpose(0, 2, 1)


def _loop_outputs(out, S: int, N: int, k_sim: int, want_Uk: bool):
    """Output arrays of a closed-loop call: fresh ones, or the caller's preallocated (e.g. pinned) ones from ``out``.
    The C ABI writes through raw addresses, so a supplied array must be exactly what the library expects --
    dtype, shape and C-contiguity are checked here instead of letting the D2H copy overrun or scramble host memory."""
    spec = dict(xk=((S, k_sim + 1, 2), np.float64), uk=((S, k_sim), np.float64), Uk=((S, k_sim, N), np.float64),
                cost=((S,), np.float64), inner_iters=((S, k_sim), np.int32), qp_iters=((S, k_sim), np.int32),
                status=((S,), np.int32))
    o = out if out is not None else {}
    res = []
    for key in ("xk", "uk", "Uk", "cost", "inner_iters", "qp_iters", "status"):
        shape, dt = spec[key]
        a = o.get(key)
        if key == "Uk" and not want_Uk:
            res.append(None)
            continue
        if a is None:
            a = np.empty(shape, dtype=dt)
        else:
            if not isinstance(a, np.ndarray) or a.dtype != dt:
                raise ValueError(f"out[{key!r}] must be a numpy array of dtype {np.dtype(dt).name}")
            if a.shape != shape:
                raise ValueError(f"out[{key!r}] has shape {a.shape}, expected {shape}")
            if not a.flags.c_contiguous or not a.flags.writeable:
                raise ValueError(f"out[{key!r}] must be C-contiguous and writeable")
        res.append(a)
    return res


def device_count() -> int:
    """Number of CUDA devices the library can see (``ntm_device_count``)."""
    n = ctypes.c_int(0)
    check(load().ntm_device_count(ctypes.byref(n)))
    return int(n.value)


def closed_loop_multi(x0, params, N: int, k_sim: int = 20, i_sim: int = 10, eps: float = 1e-14, profile: int = 0,
                      want_Uk: bool = False, out: Optional[dict] = None, state_rows: int = 0, xbounds=None,
                      devices=None):
    """``NtmMpc.closed_loop`` on several GPUs from this ONE process (``ntm_mpc_closed_loop_multi``): contiguous scenario
    shards, one pooled handle + host thread per device, shards DMA'd straight to and from the host arrays.
    ``devices``: None = every visible device, an int = the first n, or a list of ordinals."""
    x0 = _f64(x0).reshape(-1, 2)
    S = x0.shape[0]
    p = _f64(params)
    if p.ndim == 1:
        p = p.reshape(1, NPARAM)
    if p.shape not in ((1, NPARAM), (S, NPARAM)):
        raise ValueError(f"params must be [{NPARAM}] or [S,{NPARAM}], got {p.shape}")
    pc = int(p.shape[0])
    xk, uk, Uk, cost, inner, qpit, status = _loop_outputs(out, S, N, k_sim, want_Uk)
    if devices is None:
        nd, dv = 0, None
    elif isinstance(devices, int):
        nd, dv = int(devices), None
    else:
        dv = np.ascontiguousarray(devices, dtype=np.int32)
        nd = int(dv.size)
    xb = _f64(MC_STATE_BOX if xbounds is None else xbounds).reshape(4)
    check(load().ntm_mpc_closed_loop_multi(nd, _ptr(dv) if dv is not None else None, LAYOUT_MATLAB, profile, S, N, k_sim,
                                           i_sim, eps, _ptr(x0), _ptr(p), pc, int(state_rows),
                                           _ptr(xb) if state_rows else None, _ptr(xk), _ptr(uk),
                                           _ptr(Uk) if want_Uk else None, _ptr(cost), _ptr(inner), _ptr(qpit), _ptr(status)))
    return dict(xk=xk, uk=uk, Uk=Uk if want_Uk else None, cost=cost, inner_iters=inner, qp_iters=qpit, status=status)



class NtmMpc:
    """One handle = one GPU + one stream.  Not thread-safe (one per host thread)."""

    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        self._h = ctypes.c_void_p()
        check(self._lib.ntm_create(ctypes.byref(self._h), device))
        self.device = device

    # ------------------------------------------------------------------ lifetime
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.ntm_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_stream(self, cuda_stream: int) -> None:
        """``cuda_stream`` is a cudaStream_t address (e.g. ``torch.cuda.current_stream().cuda_stream``); 0 is the
        legacy default stream.  ``reset_stream()`` returns to the handle's private stream."""
        check(self._lib.ntm_set_stream(self._h, ctypes.c_void_p(cuda_stream or None)))

    def reset_stream(self) -> None:
        check(self._lib.ntm_reset_stream(self._h))

    def sync(self) -> None:
        check(self._lib.ntm_sync(self._h))

    def device_info(self) -> Dict[str, int]:
        sm, ma, mi = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        check(self._lib.ntm_device_info(self._h, ctypes.byref(sm), ctypes.byref(ma), ctypes.byref(mi)))
        return dict(sm_count=sm.value, cc_major=ma.value, cc_minor=mi.value)

    def launch_count(self) -> int:
        return int(self._lib.ntm_launch_count(self._h))

    def fp64_peak(self, iters: int = 4096):
        tf, ms = ctypes.c_double(), ctypes.c_double()
        check(self._lib.ntm_fp64_peak(self._h, iters, ctypes.byref(tf), ctypes.byref(ms)))
        return tf.value, ms.value

    def dmma_peak(self, iters: int = 4096):
        """FP64 tensor-core (DMMA.8x8x4) rate of register-resident chains: (TFLOP/s, ms)."""
        tf, ms = ctypes.c_double(), ctypes.c_double()
        check(self._lib.ntm_dmma_peak(self._h, iters, ctypes.byref(tf), ctypes.byref(ms)))
        return tf.value, ms.value

    # ------------------------------------------------------------------ helpers
    @staticmethod
    def _params(params, S: int):
        """Accepts [NPARAM] (broadcast) or [S, NPARAM]; returns (flat array, params_count)."""
        p = _f64(params)
        if p.ndim == 1:
            if p.size != NPARAM:
                raise ValueError(f"params must have {NPARAM} entries")
            return p, 1
        if p.shape != (S, NPARAM):
            raise ValueError(f"params must be [{NPARAM}] or [S,{NPARAM}] (got {p.shape}); "
                             "use params_soa.T for an SoA block")
        return p, S

    # ------------------------------------------------------------------ rho1.m, rho2.m, rho3.m
    def rho(self, x, params, profile: int = 0):
        x = _f64(x).reshape(-1, 2)
        S = x.shape[0]
        p, pc = self._params(params, S)
        r1, r2, r3 = np.empty(S), np.empty(S), np.empty(S)
        check(self._lib.ntm_rho(self._h, LAYOUT_MATLAB, profile, S, _ptr(x), _ptr(p), pc, _ptr(r1), _ptr(r2), _ptr(r3)))
        return r1, r2, r3

    # ------------------------------------------------------------------ A.m, B.m
    def lpv_AB(self, rho1, rho2, rho3, params):
        r1, r2, r3 = _f64(rho1).ravel(), _f64(rho2).ravel(), _f64(rho3).ravel()
        S = r1.size
        p, pc = self._params(params, S)
        A, B = np.empty(4 * S), np.empty(2 * S)
        check(self._lib.ntm_lpv_AB(self._h, LAYOUT_MATLAB, S, _ptr(r1), _ptr(r2), _ptr(r3), _ptr(p), pc, _ptr(A), _ptr(B)))
        return _blocks_out(A, S, 2, 2), B.reshape(S, 2)

    # ------------------------------------------------------------------ Rho_to_PhiGammaLambda.m
    def condense(self, Rho1, Rho2, Rho3, params, profile: int = 0):
        R1, R2, R3 = _f64(Rho1), _f64(Rho2), _f64(Rho3)
        if R1.ndim == 1:
            R1, R2, R3 = R1[None], R2[None], R3[None]
        S, N = R1.shape
        p, pc = self._params(params, S)
        Phi, Gam, Lam = np.empty(4 * N * S), np.empty(2 * N * N * S), np.empty(2 * N * S)
        check(self._lib.ntm_condense(self._h, LAYOUT_MATLAB, profile, S, N, _ptr(R1), _ptr(R2), _ptr(R3), _ptr(p), pc,
                                     _ptr(Phi), _ptr(Gam), _ptr(Lam)))
        return _blocks_out(Phi, S, 2 * N, 2), _blocks_out(Gam, S, 2 * N, N), Lam.reshape(S, 2 * N)

    # ------------------------------------------------------------------ NTM_MPC_Sim.m:72-73
    def hessian_grad(self, Phi, Gamma, Lambda, x, params):
        Gamma = np.asarray(Gamma, dtype=np.float64)
        if Gamma.ndim == 2:
            Gamma = Gamma[None]
        S, twoN, N = Gamma.shape
        Phi_f = _blocks_in(Phi, S, 2 * N, 2); Gam_f = _blocks_in(Gamma, S, 2 * N, N)
        Lam = _f64(Lambda).reshape(S, 2 * N); x = _f64(x).reshape(S, 2)
        p, pc = self._params(params, S)
        G, F = np.empty(N * N * S), np.empty(N * S)
        check(self._lib.ntm_hessian_grad(self._h, LAYOUT_MATLAB, S, N, _ptr(Phi_f), _ptr(Gam_f), _ptr(Lam), _ptr(x),
                                         _ptr(p), pc, _ptr(G), _ptr(F)))
        return _blocks_out(G, S, N, N), F.reshape(S, N)

    # ------------------------------------------------------------------ getWLc.m
    def getWLc(self, xmax, xmin, umax, umin, Gamma, Phi, Lambda):
        """Returns W [S, 6N+4, 2], L [S, 6N+4, N], c [S, 6N+4] of ``L U <= c + W x`` (getWLc.m, defect D9 repaired)."""
        Gamma = np.asarray(Gamma, dtype=np.float64)
        if Gamma.ndim == 2:
            Gamma = Gamma[None]
        S, twoN, N = Gamma.shape
        R = 6 * N + 4
        Gam_f = _blocks_in(Gamma, S, 2 * N, N); Phi_f = _blocks_in(Phi, S, 2 * N, 2)
        Lam = _f64(Lambda).reshape(S, 2 * N)
        b = np.array([np.ravel(xmax)[0], np.ravel(xmax)[1], np.ravel(xmin)[0], np.ravel(xmin)[1],
                      float(np.ravel(umax)[0]), float(np.ravel(umin)[0])], dtype=np.float64)
        W, L, c = np.empty(R * 2 * S), np.empty(R * N * S), np.empty(R * S)
        check(self._lib.ntm_getWLc(self._h, LAYOUT_MATLAB, S, N, _ptr(b), _ptr(Gam_f), _ptr(Phi_f), _ptr(Lam),
                                   _ptr(W), _ptr(L), _ptr(c)))
        return _blocks_out(W, S, R, 2), _blocks_out(L, S, R, N), c.reshape(S, R)

    # ------------------------------------------------------------------ quadprog, box rows only
    def qp_box(self, G, F, lb, ub):
        G = np.asarray(G, dtype=np.float64)
        if G.ndim == 2:
            G = G[None]
        S, N, _ = G.shape
        G_f = _blocks_in(G, S, N, N); F = _f64(F).reshape(S, N)
        lb, ub = np.asarray(lb, dtype=np.float64), np.asarray(ub, dtype=np.float64)
        if lb.ndim == 2 or ub.ndim == 2:
            lbf = _f64(np.broadcast_to(lb, (S, N))); ubf = _f64(np.broadcast_to(ub, (S, N))); bc = S
        else:
            lbf = _f64(np.broadcast_to(lb, (N,))); ubf = _f64(np.broadcast_to(ub, (N,))); bc = 1
        U = np.empty(N * S); it = np.empty(S, dtype=np.int32); st = np.empty(S, dtype=np.int32)
        check(self._lib.ntm_qp_box(self._h, LAYOUT_MATLAB, S, N, _ptr(G_f), _ptr(F), _ptr(lbf), _ptr(ubf), bc,
                                   _ptr(U), _ptr(it), _ptr(st)))
        return U.reshape(S, N), it, st

    # ------------------------------------------------------------------ NTM_MPC_Sim.m:97 with getWLc's state rows
    def qp_ineq(self, G, F, lb, ub, Lg, bg):
        """``min 1/2 U'GU + F'U, lb <= U <= ub, Lg U <= bg``; G [S,N,N], Lg [S,M,N], bg [S,M].  Returns
        ``(U [S,N], iters, status)``; status 3 = infeasible (quadprog exitflag -2)."""
        G = np.asarray(G, dtype=np.float64)
        if G.ndim == 2:
            G = G[None]
        S, N, _ = G.shape
        Lg = np.asarray(Lg, dtype=np.float64)
        if Lg.ndim == 2:
            Lg = np.broadcast_to(Lg, (S,) + Lg.shape)
        M = Lg.shape[1]
        if not (np.all(np.isfinite(np.asarray(lb, dtype=np.float64))) and np.all(np.isfinite(np.asarray(ub, dtype=np.float64)))):
            raise ValueError("ntm_qp_ineq needs finite lower and upper bounds on every variable")
        G_f = _blocks_in(G, S, N, N); F = _f64(F).reshape(S, N)
        L_f = _blocks_in(Lg, S, M, N) if M else np.zeros(0)
        bg = _f64(np.broadcast_to(np.asarray(bg, dtype=np.float64).reshape(-1, M) if M else np.zeros((S, 0)), (S, M)))
        lb, ub = np.asarray(lb, dtype=np.float64), np.asarray(ub, dtype=np.float64)
        if lb.ndim == 2 or ub.ndim == 2:
            lbf = _f64(np.broadcast_to(lb, (S, N))); ubf = _f64(np.broadcast_to(ub, (S, N))); bc = S
        else:
            lbf = _f64(np.broadcast_to(lb, (N,))); ubf = _f64(np.broadcast_to(ub, (N,))); bc = 1
        U = np.empty(N * S); it = np.empty(S, dtype=np.int32); st = np.empty(S, dtype=np.int32)
        check(self._lib.ntm_qp_ineq(self._h, LAYOUT_MATLAB, S, N, M, _ptr(G_f), _ptr(F), _ptr(lbf), _ptr(ubf), bc,
                                    _ptr(L_f) if M else None, _ptr(bg) if M else None, _ptr(U), _ptr(it), _ptr(st)))
        return U.reshape(S, N), it, st

    # ------------------------------------------------------------------ NTM_MPC_Sim.m:130
    def plant_step(self, x, u, params, profile: int = 0):
        x = _f64(x).reshape(-1, 2)
        S = x.shape[0]
        u = _f64(u).reshape(S)
        p, pc = self._params(params, S)
        xn = np.empty(2 * S)
        check(self._lib.ntm_plant_step(self._h, LAYOUT_MATLAB, profile, S, _ptr(x), _ptr(u), _ptr(p), pc, _ptr(xn)))
        return xn.reshape(S, 2)

    def plant_step_dev(self, S: int, profile: int, layout: int, x_ptr: int, u_ptr: int, params_ptr: int,
                       params_count: int, xn_ptr: int) -> None:
        """``plant_step`` on device pointers, asynchronous on the handle's stream (``ntm_plant_step_dev``)."""
        check(self._lib.ntm_plant_step_dev(self._h, layout, profile, S, x_ptr, u_ptr, params_ptr, params_count, xn_ptr))

    # ------------------------------------------------------------------ NTM_MPC_Sim.m:63-131, fused
    def closed_loop(self, x0, params, N: int, k_sim: int = 20, i_sim: int = 10, eps: float = 1e-14,
                    profile: int = 0, want_Uk: bool = False, out: Optional[dict] = None, state_rows: int = 0,
                    xbounds=None):
        """Host buffers in, host buffers out (H2D / D2H inside the call).  ``out`` may carry
        preallocated (e.g. pinned) arrays under the same keys to avoid allocation.

        ``state_rows`` (``STATE_ROWS_REFRESH`` / ``STATE_ROWS_FROZEN``) keeps getWLc's state rows in every QP
        (NTM_MPC_Sim.m:74,97; ``ntm_mpc_closed_loop_sc``); ``xbounds = (xmin1, xmax1, xmin2, xmax2)``, default the
        script's own state box (:39-45)."""
        x0 = _f64(x0).reshape(-1, 2)
        S = x0.shape[0]
        p, pc = self._params(params, S)
        xk, uk, Uk, cost, inner, qpit, status = _loop_outputs(out, S, N, k_sim, want_Uk)
        if state_rows:
            xb = _f64(MC_STATE_BOX if xbounds is None else xbounds).reshape(4)
            check(self._lib.ntm_mpc_closed_loop_sc(self._h, LAYOUT_MATLAB, profile, S, N, k_sim, i_sim, eps, _ptr(x0), _ptr(p),
                                                   pc, int(state_rows), _ptr(xb), _ptr(xk), _ptr(uk),
                                                   _ptr(Uk) if want_Uk else None, _ptr(cost), _ptr(inner), _ptr(qpit),
                                                   _ptr(status)))
            return dict(xk=xk, uk=uk, Uk=Uk if want_Uk else None, cost=cost, inner_iters=inner, qp_iters=qpit, status=status)
        check(self._lib.ntm_mpc_closed_loop(self._h, LAYOUT_MATLAB, profile, S, N, k_sim, i_sim, eps, _ptr(x0), _ptr(p), pc,
                                            _ptr(xk), _ptr(uk), _ptr(Uk) if want_Uk else None, _ptr(cost), _ptr(inner),
                                            _ptr(qpit), _ptr(status)))
        return dict(xk=xk, uk=uk, Uk=Uk if want_Uk else None, cost=cost, inner_iters=inner, qp_iters=qpit, status=status)

    def closed_loop_dev(self, S: int, N: int, k_sim: int, i_sim: int, eps: float, profile: int, layout: int,
                        x0_ptr: int, params_ptr: int, params_count: int, xk_ptr: int, uk_ptr: int, Uk_ptr: int = 0,
                        cost_ptr: int = 0, inner_ptr: int = 0, qp_ptr: int = 0, status_ptr: int = 0) -> None:
        """Device pointers (e.g. ``tensor.data_ptr()``); asynchronous on the handle's stream."""
        check(self._lib.ntm_mpc_closed_loop_dev(self._h, layout, profile, S, N, k_sim, i_sim, eps, x0_ptr, params_ptr,
                                                params_count, xk_ptr, uk_ptr, Uk_ptr or None, cost_ptr or None,
                                                inner_ptr or None, qp_ptr or None, status_ptr or None))

    def closed_loop_rec_dev(self, S: int, N: int, k_sim: int, i_sim: int, eps: float, profile: int, x0_ptr: int,
                            params_ptr: int, params_count: int, rec_ptr: int, inner_ptr: int = 0, qp_ptr: int = 0,
                            state_rows: int = 0, xbounds=None) -> None:
        """Resident entry writing ONE packed record [xk | uk | cost | status] of ``rec_doubles(k_sim)`` doubles per
        scenario (``ntm_mpc_closed_loop_rec_dev``): the block a multi-GPU caller gathers with a single collective."""
        xb = _f64(MC_STATE_BOX if xbounds is None else xbounds).reshape(4)
        check(self._lib.ntm_mpc_closed_loop_rec_dev(self._h, profile, S, N, k_sim, i_sim, eps, x0_ptr, params_ptr,
                                                    params_count, int(state_rows), _ptr(xb) if state_rows else None,
                                                    rec_ptr, inner_ptr or None, qp_ptr or None))

    def closed_loop_sc_dev(self, S: int, N: int, k_sim: int, i_sim: int, eps: float, profile: int, layout: int,
                           x0_ptr: int, params_ptr: int, params_count: int, state_rows: int, xbounds, xk_ptr: int,
                           uk_ptr: int, Uk_ptr: int = 0, cost_ptr: int = 0, inner_ptr: int = 0, qp_ptr: int = 0,
                           status_ptr: int = 0) -> None:
        """``closed_loop_dev`` with the state rows kept (``ntm_mpc_closed_loop_sc_dev``); ``xbounds`` is a host 4-vector."""
        xb = _f64(xbounds).reshape(4)
        check(self._lib.ntm_mpc_closed_loop_sc_dev(self._h, layout, profile, S, N, k_sim, i_sim, eps, x0_ptr, params_ptr,
                                                   params_count, int(state_rows), _ptr(xb), xk_ptr, uk_ptr, Uk_ptr or None,
                                                   cost_ptr or None, inner_ptr or None, qp_ptr or None, status_ptr or None))

    # ------------------------------------------------------------------ NTM_MPC_Sim.m:94-128, one step, no plant
    def mpc_step(self, state, x, params, N: int, i_sim: int = 10, eps: float = 1e-14, profile: int = 0,
                 want_U: bool = False):
        """One receding-horizon step for S scenarios at their measured states ``x`` [S, 2] (``ntm_mpc_step``).

        ``state`` is a C-contiguous float64 array [S, ``ctrl_doubles(N)``] updated in place; an all-zero row is a fresh
        controller (its first step runs the offline build from ``x``), so ``state[s] = 0`` restarts scenario ``s``.
        Pass the same N, profile and params on every call for the same records.  Returns a dict with ``u`` [S],
        ``U`` [S, N] (None unless ``want_U``), ``inner_iters``, ``qp_iters`` and ``status`` [S]."""
        x = _f64(x).reshape(-1, 2)
        S = x.shape[0]
        p, pc = self._params(params, S)
        if not (isinstance(state, np.ndarray) and state.dtype == np.float64 and state.shape == (S, ctrl_doubles(N))
                and state.flags.c_contiguous and state.flags.writeable):
            raise ValueError(f"state must be a writeable C-contiguous float64 array of shape {(S, ctrl_doubles(N))}")
        u = np.empty(S)
        U = np.empty((S, N)) if want_U else None
        inner, qpit, status = (np.empty(S, dtype=np.int32) for _ in range(3))
        check(self._lib.ntm_mpc_step(self._h, LAYOUT_MATLAB, profile, S, N, i_sim, eps, _ptr(x), _ptr(p), pc, _ptr(state),
                                     _ptr(u), _ptr(U), _ptr(inner), _ptr(qpit), _ptr(status)))
        return dict(u=u, U=U, inner_iters=inner, qp_iters=qpit, status=status)

    def mpc_step_dev(self, S: int, N: int, i_sim: int, eps: float, profile: int, layout: int, x_ptr: int,
                     params_ptr: int, params_count: int, state_ptr: int, u_ptr: int, U_ptr: int = 0, inner_ptr: int = 0,
                     qp_ptr: int = 0, status_ptr: int = 0) -> None:
        """``mpc_step`` on device pointers, asynchronous on the handle's stream (``ntm_mpc_step_dev``); the records
        (``ctrl_doubles(N)`` doubles per scenario, scenario slowest) stay resident."""
        check(self._lib.ntm_mpc_step_dev(self._h, layout, profile, S, N, i_sim, eps, x_ptr, params_ptr, params_count,
                                         state_ptr, u_ptr, U_ptr or None, inner_ptr or None, qp_ptr or None,
                                         status_ptr or None))

    def controller(self, params, N: int, S: Optional[int] = None, i_sim: int = 10, eps: float = 1e-14,
                   profile: int = 0) -> "Controller":
        """A ``Controller`` on this handle that owns the records of S scenarios (S from ``params`` [S, NPARAM], or given
        with one shared [NPARAM] block)."""
        return Controller(self, params, N, S, i_sim, eps, profile)

    # ------------------------------------------------------------------ Monte-Carlo back end (SURVEY 8f-3)
    def mc_stats(self, xk, uk, cost, status, params, bounds=MC_STATE_BOX, w_suppressed: float = 0.06, hist_max: float = 0.2):
        """Reduce a batch of closed-loop results ([S,k_sim+1,2], [S,k_sim], [S], [S]) on the device; returns the
        NTM_MC_NSTAT doubles documented in include/ntm_mpc.h (see `montecarlo.describe`)."""
        xk = _f64(xk); S, K1, _ = xk.shape
        K = K1 - 1
        uk = _f64(uk).reshape(S, K)
        p, pc = self._params(params, S)
        cost = None if cost is None else _f64(cost).reshape(S)
        status = None if status is None else np.ascontiguousarray(status, dtype=np.int32).reshape(S)
        b = _f64(bounds).reshape(4)
        out = np.empty(MC_NSTAT)
        check(self._lib.ntm_mc_stats(self._h, LAYOUT_MATLAB, S, K, _ptr(xk), _ptr(uk), _ptr(cost), _ptr(status), _ptr(p), pc,
                                     _ptr(b), float(w_suppressed), float(hist_max), _ptr(out)))
        return out

    def mc_stats_dev(self, S: int, k_sim: int, layout: int, xk_ptr: int, uk_ptr: int, cost_ptr: int, status_ptr: int,
                     params_ptr: int, params_count: int, out_ptr: int, bounds=MC_STATE_BOX, w_suppressed: float = 0.06,
                     hist_max: float = 0.2) -> None:
        b = _f64(bounds).reshape(4)
        check(self._lib.ntm_mc_stats_dev(self._h, layout, S, k_sim, xk_ptr, uk_ptr, cost_ptr or None, status_ptr or None,
                                         params_ptr, params_count, _ptr(b), float(w_suppressed), float(hist_max), out_ptr))

    def mc_stats_ub_dev(self, S: int, k_sim: int, layout: int, xk_ptr: int, uk_ptr: int, cost_ptr: int, status_ptr: int,
                        umin_ptr: int, umax_ptr: int, bounds_count: int, out_ptr: int, bounds=MC_STATE_BOX,
                        w_suppressed: float = 0.06, hist_max: float = 0.2) -> None:
        """``mc_stats_dev`` with the EC-power box as two compact device arrays ``umin[S]``, ``umax[S]`` (or one shared
        pair, ``bounds_count = 1``) instead of the parameter block (``ntm_mc_stats_ub_dev``)."""
        b = _f64(bounds).reshape(4)
        check(self._lib.ntm_mc_stats_ub_dev(self._h, layout, S, k_sim, xk_ptr, uk_ptr, cost_ptr or None, status_ptr or None,
                                            umin_ptr, umax_ptr, bounds_count, _ptr(b), float(w_suppressed), float(hist_max),
                                            out_ptr))

    def condense_dev(self, S: int, N: int, profile: int, layout: int, r1_ptr: int, r2_ptr: int, r3_ptr: int,
                     params_ptr: int, params_count: int, phi_ptr: int, gam_ptr: int, lam_ptr: int) -> None:
        check(self._lib.ntm_condense_dev(self._h, layout, profile, S, N, r1_ptr, r2_ptr, r3_ptr, params_ptr, params_count,
                                         phi_ptr, gam_ptr, lam_ptr))


class Controller:
    """The receding-horizon controller of NTM_MPC_Sim.m for S scenarios, in front of a plant the caller runs::

        ctl = NtmMpc(0).controller(params, N=20)
        for k in range(k_sim):
            u = ctl.step(x)              # x: measured states [S, 2]
            x = my_plant(x, u)

    Holds the per-scenario records of ``ntm_mpc_step`` (host memory) and the fixed arguments every call for them must
    repeat.  ``reset(mask)`` restarts the selected scenarios: their next step is a first step from the state it gets."""

    def __init__(self, mpc: NtmMpc, params, N: int, S: Optional[int] = None, i_sim: int = 10, eps: float = 1e-14,
                 profile: int = 0):
        p = _f64(params)
        if S is None:
            if p.ndim != 2:
                raise ValueError("S is needed with one shared parameter block")
            S = p.shape[0]
        self.mpc, self.N, self.S, self.i_sim, self.eps, self.profile = mpc, int(N), int(S), int(i_sim), float(eps), int(profile)
        self.params, _ = NtmMpc._params(p, self.S)
        self.state = np.zeros((self.S, ctrl_doubles(self.N)))
        self.last = None

    def step(self, x, want_U: bool = False) -> np.ndarray:
        """u [S] for the measured states ``x`` [S, 2]; the full result dict of ``mpc_step`` is kept in ``last``."""
        self.last = self.mpc.mpc_step(self.state, x, self.params, self.N, self.i_sim, self.eps, self.profile, want_U)
        return self.last["u"]

    def reset(self, mask=None) -> None:
        """Fresh controllers for every scenario (``mask=None``) or for those selected by a boolean / index ``mask``."""
        if mask is None:
            self.state[:] = 0.0
        else:
            self.state[np.asarray(mask)] = 0.0
