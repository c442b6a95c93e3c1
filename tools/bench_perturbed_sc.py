"""The perturbed loop with getWLc's state rows kept, fused against stepped, on one GPU (writes OUT/bench_perturbed_sc.json).

    python tools/bench_perturbed_sc.py --out DIR [--repeats 5]

BASELINE config 3 (65,536 scenarios, N = 20), inner policy fixed(10), k_sim = 20, the binding state box
(0.05, 0.16, 2000, 12000) of profiles/r05_controller_sc_bench.json, rows REFRESH and FROZEN.  The plant draws Cw from
[0.5, 2] per scenario (montecarlo.plant_batch_params), the process disturbance d and the measurement noise v are
Gaussian with std (1e-3, 30) and (5e-4, 20) (montecarlo.noise, seed 9).  Everything resident in HBM, one stream:
  perturbed_sc   ntm_mpc_closed_loop_perturbed_sc_dev: one launch for the whole run
  step_route     zeroed records + 20 x (y = x + v_k, ntm_mpc_step_sc_dev at y, ntm_plant_step_dev on the plant's block,
                 + d_k, a torch.where that holds the state of the scenarios whose step came back infeasible, a copy of u)
  sc_unperturbed ntm_mpc_closed_loop_sc_dev, nothing perturbed (the same controller against its own model)
  perturbed_box  ntm_mpc_closed_loop_perturbed_dev: the same perturbation, the box-QP controller
timed with CUDA events, the four alternated, `repeats` runs each after a warm-up of all; medians, min, max.  The step
route's u is compared with the fused one bit for bit, up to and including each scenario's infeasible step.  ntm_mc_stats of the
fused result gives the status counts and how often the true state left the box.  The card's name and power limit are
read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "mpc-ntm-control_b200"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

from bench_controller import card  # noqa: E402

K_SIM, I_SIM, EPS = 20, 10, 1e-14
CFG, S, N = 3, 65536, 20
XB = (0.05, 0.16, 2000.0, 12000.0)
PLANT_SAMPLE = {"Cw": (0.5, 2.0)}
W_STD, V_STD, NOISE_SEED = (1e-3, 30.0), (5e-4, 20.0), 9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    import torch
    import ntm_mpc
    from ntm_mpc import montecarlo, physics
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement runs on the GPU only")
    dev = torch.device("cuda:0")
    mpc = ntm_mpc.NtmMpc(0)
    stream = torch.cuda.current_stream()
    mpc.set_stream(stream.cuda_stream)
    prof = ntm_mpc.PROFILE_INNER_FIXED
    res = dict(device=torch.cuda.get_device_name(0), nvidia_smi=card(), config=CFG, S=S, N=N, k_sim=K_SIM, i_sim=I_SIM,
               profile="fixed(10)", xbounds=XB, plant_sample=PLANT_SAMPLE, w_std=W_STD, v_std=V_STD,
               noise_seed=NOISE_SEED, repeats=args.repeats, modes=[])

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record(stream)
        return e

    P, x0, _ = physics.batch_params(CFG, S=S)
    PP = montecarlo.plant_batch_params(CFG, S, None, None, PLANT_SAMPLE)
    p = torch.from_numpy(np.ascontiguousarray(P.T)).to(dev)            # MATLAB layout: one block per scenario
    pp = torch.from_numpy(np.ascontiguousarray(PP.T)).to(dev)
    x = torch.from_numpy(x0).to(dev)
    dw, dv = montecarlo.noise(S, K_SIM, W_STD, V_STD, NOISE_SEED, dev)
    d = dw.reshape(K_SIM, 2, S).permute(2, 0, 1).contiguous()          # [S, k_sim, 2]: element 2k + i per scenario
    v = dv.reshape(K_SIM, 2, S).permute(2, 0, 1).contiguous()
    xk = torch.empty((S, K_SIM + 1, 2), dtype=torch.float64, device=dev)
    uk = torch.empty((S, K_SIM), dtype=torch.float64, device=dev)
    cost = torch.empty(S, dtype=torch.float64, device=dev)
    iters = torch.empty((2, S, K_SIM), dtype=torch.int32, device=dev)
    st = torch.empty(S, dtype=torch.int32, device=dev)
    state = torch.zeros((S, ntm_mpc.ctrl_doubles(N)), dtype=torch.float64, device=dev)
    xs = [x.clone(), torch.empty_like(x)]
    y = torch.empty_like(x)
    u = torch.empty(S, dtype=torch.float64, device=dev)
    ucat = torch.empty((S, K_SIM), dtype=torch.float64, device=dev)
    sit = torch.empty((3, S), dtype=torch.int32, device=dev)
    out = lambda: (xk.data_ptr(), uk.data_ptr(), 0, cost.data_ptr(), iters[0].data_ptr(), iters[1].data_ptr(),
                   st.data_ptr())
    for mode, mname in ((ntm_mpc.STATE_ROWS_REFRESH, "REFRESH"), (ntm_mpc.STATE_ROWS_FROZEN, "FROZEN")):

        def perturbed_sc():
            mpc.closed_loop_perturbed_dev(S, N, K_SIM, I_SIM, EPS, prof, 0, x.data_ptr(), p.data_ptr(), S, pp.data_ptr(),
                                          S, 0, d.data_ptr(), v.data_ptr(), *out(), state_rows=mode, xbounds=XB)

        def perturbed_box():
            mpc.closed_loop_perturbed_dev(S, N, K_SIM, I_SIM, EPS, prof, 0, x.data_ptr(), p.data_ptr(), S, pp.data_ptr(),
                                          S, 0, d.data_ptr(), v.data_ptr(), *out())

        def sc_unperturbed():
            mpc.closed_loop_sc_dev(S, N, K_SIM, I_SIM, EPS, prof, 0, x.data_ptr(), p.data_ptr(), S, mode, XB, *out())

        def step_route():
            state.zero_()
            xs[0].copy_(x)
            for k in range(K_SIM):
                a, b = xs[k % 2], xs[(k + 1) % 2]
                torch.add(a, v[:, k], out=y)
                mpc.mpc_step_dev(S, N, I_SIM, EPS, prof, 0, y.data_ptr(), p.data_ptr(), S, state.data_ptr(), u.data_ptr(),
                                 0, sit[0].data_ptr(), sit[1].data_ptr(), sit[2].data_ptr(), state_rows=mode, xbounds=XB)
                ucat[:, k].copy_(u)
                mpc.plant_step_dev(S, 0, 0, a.data_ptr(), u.data_ptr(), pp.data_ptr(), S, b.data_ptr())
                b.add_(d[:, k])
                torch.where((sit[2] == 3)[:, None], a, b, out=b)       # infeasible: the scenario stops here

        def timed(fn):
            e0 = ev()
            fn()
            e1 = ev()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1)

        arms = dict(perturbed_sc=perturbed_sc, step_route=step_route, sc_unperturbed=sc_unperturbed,
                    perturbed_box=perturbed_box)
        for fn in arms.values():                                  # warm-up: module load, scratch allocation, caches
            timed(fn)
        ts = {k: [] for k in arms}
        for _ in range(args.repeats):
            for k, fn in arms.items():
                ts[k].append(timed(fn))
        # the fused result last: its u against the step route's, then the statistics of the true trajectories
        step_route()
        perturbed_sc()
        torch.cuda.synchronize()
        # up to and including each scenario's infeasible step: after it the step route holds the true state, but its
        # measurement x + v_k moves on, so a held scenario may step again where the fused loop has ended it
        kk = torch.arange(K_SIM, device=dev)[None, :]
        nanu = torch.isnan(uk)
        k_end = torch.where(nanu.any(1), nanu.float().argmax(1), torch.full((S,), K_SIM, device=dev))
        m = kk <= k_end[:, None]
        same = bool(torch.equal(torch.nan_to_num(ucat[m], nan=1e300), torch.nan_to_num(uk[m], nan=1e300)))
        stv = st.cpu().numpy()
        stats = mpc.mc_stats(xk.cpu().numpy(), uk.cpu().numpy(), cost.cpu().numpy(), stv, np.ascontiguousarray(P.T),
                             bounds=XB)
        desc = montecarlo.describe(stats, 0.2)

        def rate(t):
            return dict(ms_median=statistics.median(t), ms_min=min(t), ms_max=max(t), ms_all=t,
                        scenario_steps_per_s=S * K_SIM / (statistics.median(t) * 1e-3))

        med = {k: statistics.median(t) for k, t in ts.items()}
        row = dict(state_rows=mname, **{k: rate(t) for k, t in ts.items()},
                   step_route_over_perturbed_sc=med["step_route"] / med["perturbed_sc"],
                   step_route_overhead_ms=med["step_route"] - med["perturbed_sc"],
                   perturbed_sc_over_sc_unperturbed=med["perturbed_sc"] / med["sc_unperturbed"],
                   perturbed_sc_over_perturbed_box=med["perturbed_sc"] / med["perturbed_box"],
                   uk_equals_step_route=same,
                   status_counts=dict(ok=int((stv == 0).sum()), cap=int((stv == 1).sum()), nonfinite=int((stv == 2).sum()),
                                      infeasible=int((stv == 3).sum())),
                   w_outside_box_fraction=float(desc["w_outside_box_fraction"]),
                   omega_outside_box_fraction=float(desc["omega_outside_box_fraction"]),
                   state_samples_counted=int(stats[21]))
        res["modes"].append(row)
        print(json.dumps(dict((k, row[k]) for k in ("state_rows", "step_route_over_perturbed_sc", "uk_equals_step_route",
                                                      "status_counts", "w_outside_box_fraction")))
              + " " + " ".join(f"{k} {m:.1f} ms" for k, m in med.items()), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_perturbed_sc.json"), "w") as f:
        json.dump(res, f, indent=1)
    mpc.close()


if __name__ == "__main__":
    main()
