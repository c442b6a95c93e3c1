"""Controller stepping against the fused closed loop on one GPU (writes OUT/bench_controller.json).

    python tools/bench_controller.py --out DIR [--repeats 5]

For BASELINE configs 3 (65,536 x N = 20), 2 (1,024 x N = 10) and 5 (16,384 x N = 100), inner policy fixed(10), k_sim = 20,
everything resident in HBM and ordered on one stream:
  fused       ntm_mpc_closed_loop_dev: one launch for the whole run
  controller  zeroed records + 20 x (ntm_mpc_step_dev + ntm_plant_step_dev): 40 launches
timed with CUDA events, the two alternated, `repeats` runs each after a warm-up of both; reported in scenario-steps/s
(median, min, max).  One more controller run records an event after every launch and splits its time into controller
steps and plant steps.  Then the latency of the host entry (ntm_mpc_step on NumPy arrays, one scenario, copies and
synchronisation included): p50 / p99 over 200 calls after 20 warm-up calls.  The card's name and power limit are read
in the same run (nvidia-smi query, read-only)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "mpc-ntm-control_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

K_SIM, I_SIM, EPS = 20, 10, 1e-14
CONFIGS = ((3, 65536, 20), (2, 1024, 10), (5, 16384, 100))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    except Exception as e:              # the measurement does not depend on it; say so in the output
        q = [f"nvidia-smi unavailable: {e}"]
    return q


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
    res = dict(device=torch.cuda.get_device_name(0), nvidia_smi=card(), k_sim=K_SIM, i_sim=I_SIM, profile="fixed(10)",
               repeats=args.repeats, configs=[])

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record(stream)
        return e

    for cfg, S, N in CONFIGS:
        P, x0, _ = physics.batch_params(cfg, S=S)
        p = torch.from_numpy(np.ascontiguousarray(P.T)).to(dev)
        x = torch.from_numpy(x0).to(dev)
        xk = torch.empty((S, K_SIM + 1, 2), dtype=torch.float64, device=dev)
        uk = torch.empty((S, K_SIM), dtype=torch.float64, device=dev)
        cost = torch.empty(S, dtype=torch.float64, device=dev)
        iters = torch.empty((2, S, K_SIM), dtype=torch.int32, device=dev)
        st = torch.empty(S, dtype=torch.int32, device=dev)
        state = torch.zeros((S, ntm_mpc.ctrl_doubles(N)), dtype=torch.float64, device=dev)
        xs = [x.clone(), torch.empty_like(x)]
        u = torch.empty(S, dtype=torch.float64, device=dev)
        sit = torch.empty((3, S), dtype=torch.int32, device=dev)

        def fused():
            mpc.closed_loop_dev(S, N, K_SIM, I_SIM, EPS, prof, 0, x.data_ptr(), p.data_ptr(), S, xk.data_ptr(),
                                uk.data_ptr(), 0, cost.data_ptr(), iters[0].data_ptr(), iters[1].data_ptr(), st.data_ptr())

        def controller(marks=None):
            state.zero_()
            xs[0].copy_(x)
            for k in range(K_SIM):
                a, b = xs[k % 2], xs[(k + 1) % 2]
                mpc.mpc_step_dev(S, N, I_SIM, EPS, prof, 0, a.data_ptr(), p.data_ptr(), S, state.data_ptr(), u.data_ptr(),
                                 0, sit[0].data_ptr(), sit[1].data_ptr(), sit[2].data_ptr())
                if marks is not None:
                    marks.append(ev())
                mpc.plant_step_dev(S, prof, 0, a.data_ptr(), u.data_ptr(), p.data_ptr(), S, b.data_ptr())
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
        t_plant = sum(marks[2 * k + 1].elapsed_time(marks[2 * k + 2]) for k in range(K_SIM))
        same = bool(torch.equal(xs[K_SIM % 2], xk[:, K_SIM, :]))   # the controller run ends where the fused loop ends

        def rate(ts):
            return dict(ms_median=statistics.median(ts), ms_min=min(ts), ms_max=max(ts), ms_all=ts,
                        scenario_steps_per_s=S * K_SIM / (statistics.median(ts) * 1e-3))

        # host entry, one scenario: what a MATLAB / Python loop around a real plant pays per step
        Ph, xh = np.ascontiguousarray(P.T[:1]), x0[:1].copy()
        sh = np.zeros((1, ntm_mpc.ctrl_doubles(N)))
        lat = []
        for c in range(20 + args.latency_calls):
            if c % K_SIM == 0:
                sh[:] = 0.0
            t0 = time.perf_counter()
            mpc.mpc_step(sh, xh, Ph, N, I_SIM, EPS, prof)
            t1 = time.perf_counter()
            if c >= 20:
                lat.append((t1 - t0) * 1e6)
        row = dict(config=cfg, S=S, N=N, fused=rate(tf), controller=rate(tc),
                   controller_over_fused=statistics.median(tc) / statistics.median(tf),
                   controller_split_ms=dict(mpc_step=t_step, plant_step=t_plant),
                   final_state_equals_fused=same,
                   host_step_latency_us=dict(p50=float(np.percentile(lat, 50)), p99=float(np.percentile(lat, 99)),
                                             calls=len(lat)))
        res["configs"].append(row)
        print(json.dumps(dict((k, row[k]) for k in ("config", "S", "N", "controller_over_fused", "final_state_equals_fused")))
              + f" fused {row['fused']['scenario_steps_per_s']:.4g}/s controller {row['controller']['scenario_steps_per_s']:.4g}/s"
              f" host p50 {row['host_step_latency_us']['p50']:.1f} us", flush=True)
        del p, x, xk, uk, cost, iters, st, state, xs, u, sit
        torch.cuda.empty_cache()
    mpc.reset_stream()
    mpc.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_controller.json"), "w") as f:
        json.dump(res, f, indent=1)
    print("device:", res["device"], res["nvidia_smi"])


if __name__ == "__main__":
    main()
