"""State-row controller stepping against the fused state-row loop on one GPU (writes OUT/bench_controller_sc.json).

    python tools/bench_controller_sc.py --out DIR [--repeats 5]

BASELINE config 3 (65,536 scenarios, N = 20), inner policy fixed(10), k_sim = 20, getWLc's state rows kept in every QP
with the binding state box (0.05, 0.16, 2000, 12000), rows REFRESH and FROZEN; everything resident in HBM and ordered on
one stream:
  fused       ntm_mpc_closed_loop_sc_dev: one launch for the whole run
  controller  zeroed records + 20 x (ntm_mpc_step_sc_dev + ntm_plant_step_dev + a torch.where that holds the measured
              state of the scenarios whose step came back infeasible, as a caller that stops them would, and a copy of u)
timed with CUDA events, the two alternated, `repeats` runs each after a warm-up of both; reported in scenario-steps/s
(median, min, max).  controller_overhead_ms = controller - fused (medians).  A FROZEN controller step rebuilds the
frozen rows of its record (one extra G, F build per step), so FROZEN overhead - REFRESH overhead estimates that cost.
One more controller run records an event after every launch and splits its time into controller steps and the rest.
Then the latency of the host entry (ntm_mpc_step_sc on NumPy arrays, one feasible scenario, copies and synchronisation
included): p50 / p99 over 200 calls after 20 warm-up calls.  The card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "mpc-ntm-control_b200"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

from bench_controller import card  # noqa: E402

K_SIM, I_SIM, EPS = 20, 10, 1e-14
CFG, S, N = 3, 65536, 20
XB = (0.05, 0.16, 2000.0, 12000.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--latency-calls", type=int, default=200)
    args = ap.parse_args()
    import torch
    import ntm_mpc
    from ntm_mpc import physics
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement runs on the GPU only")
    dev = torch.device("cuda:0")
    mpc = ntm_mpc.NtmMpc(0)
    stream = torch.cuda.current_stream()
    mpc.set_stream(stream.cuda_stream)
    prof = ntm_mpc.PROFILE_INNER_FIXED
    res = dict(device=torch.cuda.get_device_name(0), nvidia_smi=card(), config=CFG, S=S, N=N, k_sim=K_SIM, i_sim=I_SIM,
               profile="fixed(10)", xbounds=XB, repeats=args.repeats, modes=[])

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record(stream)
        return e

    P, x0, _ = physics.batch_params(CFG, S=S)
    p = torch.from_numpy(np.ascontiguousarray(P.T)).to(dev)
    x = torch.from_numpy(x0).to(dev)
    xk = torch.empty((S, K_SIM + 1, 2), dtype=torch.float64, device=dev)
    uk = torch.empty((S, K_SIM), dtype=torch.float64, device=dev)
    iters = torch.empty((2, S, K_SIM), dtype=torch.int32, device=dev)
    st = torch.empty(S, dtype=torch.int32, device=dev)
    state = torch.zeros((S, ntm_mpc.ctrl_doubles(N)), dtype=torch.float64, device=dev)
    xs = [x.clone(), torch.empty_like(x)]
    u = torch.empty(S, dtype=torch.float64, device=dev)
    ucat = torch.empty((S, K_SIM), dtype=torch.float64, device=dev)
    sit = torch.empty((3, S), dtype=torch.int32, device=dev)
    for mode, mname in ((ntm_mpc.STATE_ROWS_REFRESH, "REFRESH"), (ntm_mpc.STATE_ROWS_FROZEN, "FROZEN")):

        def fused():
            mpc.closed_loop_sc_dev(S, N, K_SIM, I_SIM, EPS, prof, 0, x.data_ptr(), p.data_ptr(), S, mode, XB,
                                   xk.data_ptr(), uk.data_ptr(), 0, 0, iters[0].data_ptr(), iters[1].data_ptr(),
                                   st.data_ptr())

        def controller(marks=None):
            state.zero_()
            xs[0].copy_(x)
            for k in range(K_SIM):
                a, b = xs[k % 2], xs[(k + 1) % 2]
                mpc.mpc_step_dev(S, N, I_SIM, EPS, prof, 0, a.data_ptr(), p.data_ptr(), S, state.data_ptr(), u.data_ptr(),
                                 0, sit[0].data_ptr(), sit[1].data_ptr(), sit[2].data_ptr(), state_rows=mode, xbounds=XB)
                if marks is not None:
                    marks.append(ev())
                ucat[:, k].copy_(u)
                mpc.plant_step_dev(S, prof, 0, a.data_ptr(), u.data_ptr(), p.data_ptr(), S, b.data_ptr())
                torch.where((sit[2] == 3)[:, None], a, b, out=b)       # infeasible: the scenario stops here
                if marks is not None:
                    marks.append(ev())

        def timed(fn):
            e0 = ev()
            fn()
            e1 = ev()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1)

        timed(fused); timed(controller)                           # warm-up: module load, scratch allocation, caches
        tf, tc = [], []
        for _ in range(args.repeats):
            tf.append(timed(fused)); tc.append(timed(controller))
        marks = [ev()]
        controller(marks)
        torch.cuda.synchronize()
        t_step = sum(marks[2 * k].elapsed_time(marks[2 * k + 1]) for k in range(K_SIM))
        t_rest = sum(marks[2 * k + 1].elapsed_time(marks[2 * k + 2]) for k in range(K_SIM))
        # the controller run gives the fused loop's inputs bit for bit, NaN from the infeasible step on included
        same = bool(torch.allclose(ucat, uk, rtol=0.0, atol=0.0, equal_nan=True))
        stv = st.cpu().numpy()

        def rate(ts):
            return dict(ms_median=statistics.median(ts), ms_min=min(ts), ms_max=max(ts), ms_all=ts,
                        scenario_steps_per_s=S * K_SIM / (statistics.median(ts) * 1e-3))

        # host entry, one scenario that stays feasible over the run
        s1 = int(np.flatnonzero(stv == 0)[0])
        Ph, xh = np.ascontiguousarray(P.T[s1:s1 + 1]), x0[s1:s1 + 1].copy()
        sh = np.zeros((1, ntm_mpc.ctrl_doubles(N)))
        lat = []
        for c in range(20 + args.latency_calls):
            if c % K_SIM == 0:
                sh[:] = 0.0
            t0 = time.perf_counter()
            mpc.mpc_step(sh, xh, Ph, N, I_SIM, EPS, prof, state_rows=mode, xbounds=XB)
            t1 = time.perf_counter()
            if c >= 20:
                lat.append((t1 - t0) * 1e6)
        row = dict(state_rows=mname, fused=rate(tf), controller=rate(tc),
                   controller_over_fused=statistics.median(tc) / statistics.median(tf),
                   controller_overhead_ms=statistics.median(tc) - statistics.median(tf),
                   controller_split_ms=dict(mpc_step_sc=t_step, plant_and_hold=t_rest),
                   uk_equals_fused=same, fused_status_counts=dict(ok=int((stv == 0).sum()), cap=int((stv == 1).sum()),
                                                                  nonfinite=int((stv == 2).sum()),
                                                                  infeasible=int((stv == 3).sum())),
                   host_step_latency_us=dict(p50=float(np.percentile(lat, 50)), p99=float(np.percentile(lat, 99)),
                                             calls=len(lat), scenario=s1))
        res["modes"].append(row)
        print(json.dumps(dict((k, row[k]) for k in ("state_rows", "controller_over_fused", "controller_overhead_ms",
                                                      "uk_equals_fused")))
              + f" fused {row['fused']['ms_median']:.1f} ms controller {row['controller']['ms_median']:.1f} ms"
              f" host p50 {row['host_step_latency_us']['p50']:.1f} us", flush=True)
    m = {r["state_rows"]: r for r in res["modes"]}
    res["frozen_row_rebuild_ms_per_run_estimate"] = m["FROZEN"]["controller_overhead_ms"] - m["REFRESH"]["controller_overhead_ms"]
    mpc.reset_stream()
    mpc.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_controller_sc.json"), "w") as f:
        json.dump(res, f, indent=1)
    print("device:", res["device"], res["nvidia_smi"])


if __name__ == "__main__":
    main()
