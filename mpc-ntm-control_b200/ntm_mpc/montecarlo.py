"""Monte-Carlo front and back end around the fused closed loop (SURVEY 8f-3): scenario batches in (the samplers of
``physics.make_batch``: BASELINE configs 2-5), statistics and trajectory files out.

``run`` keeps everything on the GPU between the loop and the reduction: H2D of x0/params, ``ntm_mpc_closed_loop_dev``,
``ntm_mc_stats_dev`` on the same stream, D2H of NTM_MC_NSTAT doubles (and of the trajectories only when asked for).
Writers: ``.npz`` (numpy) and MATLAB ``.mat`` v7 (scipy.io) with the variable names the script leaves in its workspace
(``xk``, ``uk``, NTM_MPC_Sim.m:82-84) so that the plotting cells :137-161 run on a loaded file."""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np

from . import physics
from ._lib import LAYOUT_SOA, NPARAM
from .api import MC_NBINS, MC_NSTAT, MC_STATE_BOX, PLANT_PROFILE_BITS, NtmMpc


def describe(stats: np.ndarray, hist_max: float = 0.2) -> Dict[str, object]:
    """Names for the NTM_MC_NSTAT doubles of ``ntm_mc_stats`` (include/ntm_mpc.h) plus the derived means."""
    s = np.asarray(stats, dtype=np.float64)
    n = s[0] + s[1]                                          # scenarios that entered the sums: the kernel leaves out every status >= NTM_SCN_NONFINITE (non-finite AND infeasible)
    d = {
        "scenarios_ok": int(s[0]), "scenarios_iter_cap": int(s[1]), "scenarios_nonfinite": int(s[2]),
        "scenarios_infeasible": int(s[3]),
        "cost_mean": s[4] / n if n else float("nan"), "cost_min": s[6], "cost_max": s[7],
        "cost_std": float(np.sqrt(max(s[5] / n - (s[4] / n) ** 2, 0.0))) if n else float("nan"),
        "w_final_mean": s[8] / n if n else float("nan"), "w_final_min": s[10], "w_final_max": s[11],
        "w_final_std": float(np.sqrt(max(s[9] / n - (s[8] / n) ** 2, 0.0))) if n else float("nan"),
        "suppressed_fraction": s[12] / n if n else float("nan"),
        "steps_to_suppression_mean": s[13] / s[14] if s[14] else float("nan"),
        "reached_suppression_fraction": s[14] / n if n else float("nan"),
        "u_at_umin_fraction": s[15] / s[17] if s[17] else float("nan"),
        "u_at_umax_fraction": s[16] / s[17] if s[17] else float("nan"),
        "active_bound_fraction": (s[15] + s[16]) / s[17] if s[17] else float("nan"),
        "u_mean": s[18] / s[17] if s[17] else float("nan"),
        "w_outside_box_fraction": s[19] / s[21] if s[21] else float("nan"),
        "omega_outside_box_fraction": s[20] / s[21] if s[21] else float("nan"),
        "w_final_hist": s[22:22 + MC_NBINS].astype(np.int64),
        "w_final_hist_edges": np.linspace(0.0, hist_max, MC_NBINS + 1),
    }
    return d


def run(config: int = 3, S: Optional[int] = None, seed: Optional[int] = None, profile: int = 0, k_sim: int = 20,
        i_sim: int = 10, eps: float = 1e-14, bounds=MC_STATE_BOX, w_suppressed: float = 0.06, hist_max: float = 0.2,
        trajectories: bool = False, handle: Optional[NtmMpc] = None, device: int = 0,
        state_rows: int = 0, sample=None, plant_sample=None, plant_profile: Optional[int] = None, w_std=None,
        v_std=None, noise_seed: Optional[int] = None) -> Dict[str, object]:
    """One Monte-Carlo batch of BASELINE config ``config`` through the fused loop; returns ``describe(...)`` of the
    on-device reduction, ``N``, ``S`` and -- with ``trajectories`` -- ``xk [S,k_sim+1,2]``, ``uk [S,k_sim]``,
    ``cost [S]``, ``status [S]`` on the host.  ``state_rows`` != 0 keeps getWLc's state rows (box = ``bounds``) in every
    QP (``ntm_mpc_closed_loop_sc_dev``); infeasible scenarios are counted in ``stats[3]`` and left out of the moments.
    ``sample`` = ``{name: (lo, hi)}``: extra physics entries drawn per scenario (``physics.make_batch``), e.g. the
    constants the authors flag as unknown: ``{"Cw": (0.5, 2.0)}`` (NTM_MPC_Sim.m:19), ``{"c_tauE": (0.0, 1.5)}`` with
    ``profile | PROFILE_TAUE_W`` (:14).  Those draws change the controller's model together with the plant.

    Robustness (``ntm_mpc_closed_loop_perturbed_dev``): with any of ``plant_sample``, ``plant_profile``, ``w_std``,
    ``v_std`` the controller keeps the block above while the plant gets the same block with the ``plant_sample``
    entries redrawn per scenario (``plant_batch_params``), e.g. ``{"Cw": (0.5, 2.0)}``: a nominal controller against
    plants with unknown ``Cw``; ``{"c_tauE": ...}`` with ``plant_profile=PROFILE_TAUE_W``: constant tau_E in the
    controller, tau_E(w) in the plant.  ``plant_profile`` defaults to the plant bits of ``profile``.  ``w_std`` /
    ``v_std`` (scalar or per-component pair): Gaussian process disturbances d_k and measurement noise v_k, drawn on the
    device by ``noise`` and never copied to the host.  The reduction runs on the true trajectories with the controller's
    umin / umax.  Not combined with ``state_rows``."""
    import torch                                               # device buffers + stream plumbing only
    h = handle or NtmMpc(device)
    prm, x0, N = physics.batch_params(config, S, seed, sample) # [NPARAM, S] SoA, [S, 2]
    S = x0.shape[0]
    perturbed = plant_sample is not None or plant_profile is not None or w_std is not None or v_std is not None
    if perturbed and state_rows:
        raise ValueError("the perturbed plant runs the box-QP controller: state_rows must be 0")
    dev = torch.device(f"cuda:{device}")
    d_prm = torch.from_numpy(prm).to(dev)                      # SoA block: scenario index fastest
    d_x0 = torch.from_numpy(np.ascontiguousarray(x0.T)).to(dev)
    d_xk = torch.empty(2 * (k_sim + 1) * S, dtype=torch.float64, device=dev)
    d_uk = torch.empty(k_sim * S, dtype=torch.float64, device=dev)
    d_cost = torch.empty(S, dtype=torch.float64, device=dev)
    d_st = torch.empty(S, dtype=torch.int32, device=dev)
    d_out = torch.empty(MC_NSTAT, dtype=torch.float64, device=dev)
    h.set_stream(torch.cuda.current_stream(dev).cuda_stream or None)
    try:
        if perturbed:
            pf = (profile & PLANT_PROFILE_BITS) if plant_profile is None else int(plant_profile)
            d_pp = torch.from_numpy(plant_batch_params(config, S, seed, sample, plant_sample)).to(dev) \
                if plant_sample else None
            d_w, d_v = noise(S, k_sim, w_std, v_std, noise_seed, dev)
            h.closed_loop_perturbed_dev(S, N, k_sim, i_sim, eps, profile, LAYOUT_SOA, d_x0.data_ptr(), d_prm.data_ptr(), S,
                                        d_pp.data_ptr() if d_pp is not None else 0, S, pf,
                                        d_w.data_ptr() if d_w is not None else 0, d_v.data_ptr() if d_v is not None else 0,
                                        d_xk.data_ptr(), d_uk.data_ptr(), 0, d_cost.data_ptr(), 0, 0, d_st.data_ptr())
        elif state_rows:
            h.closed_loop_sc_dev(S, N, k_sim, i_sim, eps, profile, LAYOUT_SOA, d_x0.data_ptr(), d_prm.data_ptr(), S,
                                 state_rows, bounds, d_xk.data_ptr(), d_uk.data_ptr(), 0, d_cost.data_ptr(), 0, 0,
                                 d_st.data_ptr())
        else:
            h.closed_loop_dev(S, N, k_sim, i_sim, eps, profile, LAYOUT_SOA, d_x0.data_ptr(), d_prm.data_ptr(), S,
                              d_xk.data_ptr(), d_uk.data_ptr(), 0, d_cost.data_ptr(), 0, 0, d_st.data_ptr())
        h.mc_stats_dev(S, k_sim, LAYOUT_SOA, d_xk.data_ptr(), d_uk.data_ptr(), d_cost.data_ptr(), d_st.data_ptr(),
                       d_prm.data_ptr(), S, d_out.data_ptr(), bounds, w_suppressed, hist_max)
        stats = d_out.cpu().numpy()
    finally:
        h.reset_stream()
        if handle is None:
            h.close()
    res = describe(stats, hist_max)
    res.update(config=config, S=S, N=N, k_sim=k_sim, profile=profile, state_rows=state_rows, stats=stats)
    if perturbed:
        res.update(plant_profile=pf, w_std=np.zeros(2) if w_std is None else np.broadcast_to(np.asarray(w_std, float), (2,)),
                   v_std=np.zeros(2) if v_std is None else np.broadcast_to(np.asarray(v_std, float), (2,)))
        if plant_sample:
            res["plant_params"] = d_pp.cpu().numpy()
    if trajectories:
        res["xk"] = np.ascontiguousarray(d_xk.cpu().numpy().reshape(2 * (k_sim + 1), S).T.reshape(S, k_sim + 1, 2))
        res["uk"] = np.ascontiguousarray(d_uk.cpu().numpy().reshape(k_sim, S).T)
        res["cost"] = d_cost.cpu().numpy(); res["status"] = d_st.cpu().numpy()
    return res


def plant_batch_params(config: int, S: int, seed: Optional[int], sample, plant_sample) -> np.ndarray:
    """The plant's ``[NPARAM, S]`` SoA block for ``run``: ``physics.make_batch(config, S, seed, sample)`` with the
    ``plant_sample`` entries drawn uniformly per scenario from their OWN generator (PCG64(seed + 2), one column per name
    in sorted order), so the controller's block and the base batch are unchanged by the option."""
    phys, _, _ = physics.make_batch(config, S, seed, sample)
    Sfull = physics.CONFIG_SHAPES[config][0]
    rng = np.random.Generator(np.random.PCG64((Sfull if seed is None else seed) + 2))
    u = rng.random((S, len(plant_sample)))
    for c, key in enumerate(sorted(plant_sample)):
        if key not in phys:
            raise KeyError(f"unknown physics entry {key!r}")
        lo, hi = plant_sample[key]
        phys[key] = lo + (hi - lo) * u[:, c]
    return np.ascontiguousarray(physics.params_from_physics(phys).reshape(NPARAM, -1))


def noise(S: int, k_sim: int, w_std, v_std, seed: Optional[int], device):
    """``(d, v)`` for ``run``: SoA device tensors of 2 * k_sim doubles per scenario (element 2k + i, scenario fastest),
    or None where the standard deviation is None.  One ``torch.Generator(device)`` seeded with ``seed`` (default 0)
    draws ``torch.randn(k_sim, 2, S)`` for d first, then for v; each is scaled by its per-component std."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(0 if seed is None else int(seed))
    out = []
    for std in (w_std, v_std):
        if std is None:
            out.append(None)
            continue
        sd = torch.as_tensor(np.broadcast_to(np.asarray(std, dtype=np.float64), (2,)).copy(), device=device)
        z = torch.randn(k_sim, 2, S, generator=g, dtype=torch.float64, device=device)
        out.append((z * sd.view(1, 2, 1)).reshape(-1))
    return out[0], out[1]


def save_npz(path: str, result: Dict[str, object]) -> None:
    np.savez_compressed(path, **{k: np.asarray(v) for k, v in result.items()})


def save_mat(path: str, result: Dict[str, object], scenario: Optional[int] = None) -> None:
    """MATLAB v7 file.  With ``scenario`` the trajectories of that one scenario are stored under the script's own
    names and shapes (``xk`` 2 x (k_sim+1), ``uk`` 1 x k_sim, NTM_MPC_Sim.m:82-83); otherwise the whole batch
    (``xk`` 2 x (k_sim+1) x S, ``uk`` k_sim x S) plus the statistics."""
    from scipy.io import savemat
    out = {k: np.asarray(v) for k, v in result.items() if k not in ("xk", "uk")}
    if "xk" in result:
        xk = np.asarray(result["xk"]); uk = np.asarray(result["uk"])
        if scenario is not None:
            out["xk"] = xk[scenario].T; out["uk"] = uk[scenario][None, :]
        else:
            out["xk"] = xk.transpose(2, 1, 0); out["uk"] = uk.T
    savemat(path, out, do_compression=True)
