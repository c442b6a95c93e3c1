"""The observed loop (a Kalman filter between the sensor and the controller) on one GPU: cost against the perturbed loop
and the step route, the filter step alone, and what the observer changes (writes OUT/bench_observed.json).

    python tools/bench_observed.py --out DIR [--repeats 5]

1. Timing, inner policy fixed(10), k_sim = 20, box-QP controller, config 3 (65,536 scenarios, N = 20) and config 5
   (16,384, N = 100).  The plant draws Cw from [0.5, 2] per scenario (montecarlo.plant_batch_params); d and v are
   Gaussian with std (1e-3, 30) and (5e-4, 20) (montecarlo.noise, seed 9); kf_cov = kf_cov_from_std of the same.
   Everything resident in HBM, one stream:
     observed     ntm_mpc_closed_loop_observed_dev: one launch for the whole run
     perturbed    ntm_mpc_closed_loop_perturbed_dev on the same draws (the controller sees y_k)
     step_route   zeroed records + 20 x (y = x + v_k, ntm_kf_step_dev, ntm_mpc_step_dev at xhat, ntm_plant_step_dev
                  + d_k, a copy of u)
   CUDA events, the three alternated, `repeats` runs each after a warm-up of all; medians, min, max.  The step route's
   u and xhat are compared with the fused ones bit for bit.
2. ntm_kf_step_dev alone at 1,048,576 scenarios (SoA, one parameter block per scenario, resumed records) against its
   algorithmic bytes: y 16, u 8, the 8 parameters the model reads 64, the record read and written 2 x 48, xhat 16 =
   200 B per scenario; 210 MB per call, more than the 126 MB of L2.  Share of the 7.7 TB/s HBM peak of the data sheet.
3. What the observer changes, config 3 with the state rows REFRESH and FROZEN in the box (0.05, 0.16, 2000, 12000), the
   same plant and noise: infeasible scenarios, w_outside_box_fraction and mean cost of montecarlo.run with raw y
   (no kf_cov) and with kf_cov_from_std.
The card's name and power limit are read in the same run."""
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
CONFIGS = ((3, 65536, 20), (5, 16384, 100))
XB = (0.05, 0.16, 2000.0, 12000.0)
PLANT_SAMPLE = {"Cw": (0.5, 2.0)}
W_STD, V_STD, NOISE_SEED = (1e-3, 30.0), (5e-4, 20.0), 9
KF_S = 1 << 20
KF_BYTES = 16 + 8 + 64 + 2 * 48 + 16
HBM_PEAK = 7.7e12


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
    kc = montecarlo.kf_cov_from_std(W_STD, V_STD)
    res = dict(device=torch.cuda.get_device_name(0), nvidia_smi=card(), k_sim=K_SIM, i_sim=I_SIM, profile="fixed(10)",
               plant_sample=PLANT_SAMPLE, w_std=W_STD, v_std=V_STD, noise_seed=NOISE_SEED, kf_cov=kc.tolist(),
               repeats=args.repeats, loops=[])

    def timed(fn):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def rate(t, S):
        return dict(ms_median=statistics.median(t), ms_min=min(t), ms_max=max(t), ms_all=t,
                    scenario_steps_per_s=S * K_SIM / (statistics.median(t) * 1e-3))

    # ---- 1. the loop: observed, perturbed, step route
    for cfg, S, N in CONFIGS:
        P, x0, _ = physics.batch_params(cfg, S=S)
        PP = montecarlo.plant_batch_params(cfg, S, None, None, PLANT_SAMPLE)
        p = torch.from_numpy(np.ascontiguousarray(P.T)).to(dev)            # MATLAB layout: one block per scenario
        pp = torch.from_numpy(np.ascontiguousarray(PP.T)).to(dev)
        x = torch.from_numpy(x0).to(dev)
        dw, dv = montecarlo.noise(S, K_SIM, W_STD, V_STD, NOISE_SEED, dev)
        d = dw.reshape(K_SIM, 2, S).permute(2, 0, 1).contiguous()          # [S, k_sim, 2]: element 2k + i per scenario
        v = dv.reshape(K_SIM, 2, S).permute(2, 0, 1).contiguous()
        f64 = dict(dtype=torch.float64, device=dev)
        xk = torch.empty((S, K_SIM + 1, 2), **f64); uk = torch.empty((S, K_SIM), **f64)
        xhat = torch.empty((S, K_SIM, 2), **f64); cost = torch.empty(S, **f64)
        iters = torch.empty((2, S, K_SIM), dtype=torch.int32, device=dev)
        st = torch.empty(S, dtype=torch.int32, device=dev)
        state = torch.zeros((S, ntm_mpc.ctrl_doubles(N)), **f64)
        kfs = torch.zeros((S, ntm_mpc.kf_doubles()), **f64)
        xs = [x.clone(), torch.empty_like(x)]
        y = torch.empty_like(x); xh = torch.empty_like(x)
        u = torch.zeros(S, **f64)
        ucat = torch.empty((S, K_SIM), **f64); hcat = torch.empty((S, K_SIM, 2), **f64)
        sit = torch.empty((3, S), dtype=torch.int32, device=dev)
        out = lambda: (xk.data_ptr(), uk.data_ptr(), 0, cost.data_ptr(), iters[0].data_ptr(), iters[1].data_ptr(),
                       st.data_ptr())
        base = (S, N, K_SIM, I_SIM, EPS, prof, 0, x.data_ptr(), p.data_ptr(), S, pp.data_ptr(), S, 0, d.data_ptr(),
                v.data_ptr())

        def observed():
            mpc.closed_loop_observed_dev(*base, *out(), kf_cov=kc, xhat_ptr=xhat.data_ptr())

        def perturbed():
            mpc.closed_loop_perturbed_dev(*base, *out())

        def step_route():
            state.zero_(); kfs.zero_(); u.zero_()
            xs[0].copy_(x)
            for k in range(K_SIM):
                a, b = xs[k % 2], xs[(k + 1) % 2]
                torch.add(a, v[:, k], out=y)
                mpc.kf_step_dev(S, prof, 0, y.data_ptr(), u.data_ptr(), p.data_ptr(), S, kc, kfs.data_ptr(), xh.data_ptr())
                hcat[:, k].copy_(xh)
                mpc.mpc_step_dev(S, N, I_SIM, EPS, prof, 0, xh.data_ptr(), p.data_ptr(), S, state.data_ptr(), u.data_ptr(),
                                 0, sit[0].data_ptr(), sit[1].data_ptr(), sit[2].data_ptr())
                ucat[:, k].copy_(u)
                mpc.plant_step_dev(S, 0, 0, a.data_ptr(), u.data_ptr(), pp.data_ptr(), S, b.data_ptr())
                b.add_(d[:, k])

        arms = dict(observed=observed, perturbed=perturbed, step_route=step_route)
        for fn in arms.values():                                  # warm-up: module load, scratch allocation, caches
            timed(fn)
        ts = {k: [] for k in arms}
        for _ in range(args.repeats):
            for k, fn in arms.items():
                ts[k].append(timed(fn))
        step_route()
        observed()
        torch.cuda.synchronize()
        same_u = bool(torch.equal(ucat.view(torch.int64), uk.view(torch.int64)))
        same_h = bool(torch.equal(hcat.view(torch.int64), xhat.view(torch.int64)))
        med = {k: statistics.median(t) for k, t in ts.items()}
        row = dict(config=cfg, S=S, N=N, **{k: rate(t, S) for k, t in ts.items()},
                   observed_over_perturbed=med["observed"] / med["perturbed"],
                   step_route_over_observed=med["step_route"] / med["observed"],
                   uk_equals_step_route=same_u, xhat_equals_step_route=same_h)
        res["loops"].append(row)
        print(json.dumps(dict((k, row[k]) for k in ("config", "observed_over_perturbed", "step_route_over_observed",
                                                      "uk_equals_step_route", "xhat_equals_step_route")))
              + " " + " ".join(f"{k} {m:.2f} ms" for k, m in med.items()), flush=True)
        del p, pp, x, d, v, xk, uk, xhat, cost, iters, st, state, kfs, xs, ucat, hcat
        torch.cuda.empty_cache()

    # ---- 2. the filter step alone
    rng = np.random.default_rng(1)
    P, x0, _ = physics.batch_params(3, S=65536)
    reps = KF_S // 65536
    p = torch.from_numpy(np.ascontiguousarray(np.tile(P, (1, reps)))).to(dev)          # SoA [NPARAM, S]
    yk = torch.from_numpy(np.ascontiguousarray(np.tile(x0.T, (1, reps)) + rng.normal(size=(2, KF_S)) * 1e-3)).to(dev)
    uu = torch.from_numpy(rng.uniform(0.0, 2e6, size=KF_S)).to(dev)
    rec = torch.zeros((KF_S, ntm_mpc.kf_doubles()), dtype=torch.float64, device=dev)
    xo = torch.empty(2 * KF_S, dtype=torch.float64, device=dev)

    def kf():
        mpc.kf_step_dev(KF_S, prof, 1, yk.data_ptr(), uu.data_ptr(), p.data_ptr(), KF_S, kc, rec.data_ptr(), xo.data_ptr())

    for _ in range(3):                                           # warm-up; the records are resumed from here on
        timed(kf)
    reps_t = [timed(lambda: [kf() for _ in range(20)]) / 20 for _ in range(args.repeats)]
    t = statistics.median(reps_t)
    res["kf_step"] = dict(S=KF_S, layout="SoA", params_count=KF_S, bytes_per_scenario=KF_BYTES, us_median=t * 1e3,
                          us_all=[r * 1e3 for r in reps_t], achieved_TBps=KF_S * KF_BYTES / (t * 1e-3) / 1e12,
                          fraction_of_hbm_peak=KF_S * KF_BYTES / (t * 1e-3) / HBM_PEAK)
    print(json.dumps(res["kf_step"]), flush=True)
    del p, yk, uu, rec, xo
    torch.cuda.empty_cache()

    # ---- 3. what the observer changes
    res["effect"] = []
    for mode, mname in ((ntm_mpc.STATE_ROWS_REFRESH, "REFRESH"), (ntm_mpc.STATE_ROWS_FROZEN, "FROZEN")):
        for obs in (False, True):
            r = montecarlo.run(config=3, profile=prof, k_sim=K_SIM, handle=mpc, state_rows=mode, bounds=XB,
                               plant_sample=PLANT_SAMPLE, w_std=W_STD, v_std=V_STD, noise_seed=NOISE_SEED,
                               kf_cov=kc if obs else None)
            row = dict(state_rows=mname, controller_sees="xhat (kf_cov_from_std)" if obs else "y (raw)",
                       infeasible=r["scenarios_infeasible"], ok=r["scenarios_ok"], iter_cap=r["scenarios_iter_cap"],
                       nonfinite=r["scenarios_nonfinite"], w_outside_box_fraction=float(r["w_outside_box_fraction"]),
                       omega_outside_box_fraction=float(r["omega_outside_box_fraction"]), cost_mean=float(r["cost_mean"]))
            res["effect"].append(row)
            print(json.dumps(row), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_observed.json"), "w") as f:
        json.dump(res, f, indent=1)
    mpc.close()


if __name__ == "__main__":
    main()
