"""The fused loop against a perturbed plant on one GPU (writes OUT/bench_perturbed.json).

    python tools/bench_perturbed.py --out DIR [--repeats 5]

For BASELINE configs 3 (65,536 x N = 20) and 5 (16,384 x N = 100), inner policy fixed(10), k_sim = 20, everything
resident in HBM and ordered on one stream, four arms:
  a  fused         ntm_mpc_closed_loop_dev, the headline loop (Euler plant = the controller's model)
  b  fused_rk4     the same with NTM_PROFILE_PLANT_RK4: the existing cold-plant instantiation
  c  perturbed     ntm_mpc_closed_loop_perturbed_dev: nominal controller, plant with Cw drawn from U[0.5, 2.0] and the
                   RK4 integrator, Gaussian d_k and v_k: one launch
  d  step_api      zeroed records + 20 x (y = x + v_k, ntm_mpc_step_dev, ntm_plant_step_dev, x += d_k): the same run
                   through the step API, 40 library launches plus 40 element-wise adds
timed with CUDA events, the four alternated, `repeats` runs each after a warm-up of all; reported in scenario-steps/s
(median, min, max).  c and d must end on the same bits (checked, reported).  The card's name and power limit are read
in the same run (nvidia-smi query, read-only)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "mpc-ntm-control_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

K_SIM, I_SIM, EPS = 20, 10, 1e-14
CONFIGS = ((3, 65536, 20), (5, 16384, 100))
W_STD, V_STD = (1e-3, 30.0), (5e-4, 20.0)


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
    prof, rk4 = ntm_mpc.PROFILE_INNER_FIXED, ntm_mpc.PROFILE_PLANT_RK4
    res = dict(device=torch.cuda.get_device_name(0), nvidia_smi=card(), k_sim=K_SIM, i_sim=I_SIM, profile="fixed(10)",
               plant="Cw ~ U[0.5, 2.0], RK4", w_std=W_STD, v_std=V_STD, repeats=args.repeats, configs=[])

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record(stream)
        return e

    for cfg, S, N in CONFIGS:
        P, x0, _ = physics.batch_params(cfg, S=S)
        PP = montecarlo.plant_batch_params(cfg, S, None, None, {"Cw": (0.5, 2.0)})
        p = torch.from_numpy(np.ascontiguousarray(P.T)).to(dev)
        pp = torch.from_numpy(np.ascontiguousarray(PP.T)).to(dev)
        x = torch.from_numpy(x0).to(dev)
        g = torch.Generator(device=dev)
        g.manual_seed(cfg)
        d = torch.randn((S, K_SIM, 2), generator=g, dtype=torch.float64, device=dev) * torch.tensor(W_STD, device=dev)
        v = torch.randn((S, K_SIM, 2), generator=g, dtype=torch.float64, device=dev) * torch.tensor(V_STD, device=dev)
        xk = torch.empty((S, K_SIM + 1, 2), dtype=torch.float64, device=dev)
        uk = torch.empty((S, K_SIM), dtype=torch.float64, device=dev)
        cost = torch.empty(S, dtype=torch.float64, device=dev)
        iters = torch.empty((2, S, K_SIM), dtype=torch.int32, device=dev)
        st = torch.empty(S, dtype=torch.int32, device=dev)
        state = torch.zeros((S, ntm_mpc.ctrl_doubles(N)), dtype=torch.float64, device=dev)
        xs = [x.clone(), torch.empty_like(x)]
        y = torch.empty_like(x)
        u = torch.empty(S, dtype=torch.float64, device=dev)
        sit = torch.empty((3, S), dtype=torch.int32, device=dev)

        def loop(profile):
            mpc.closed_loop_dev(S, N, K_SIM, I_SIM, EPS, profile, 0, x.data_ptr(), p.data_ptr(), S, xk.data_ptr(),
                                uk.data_ptr(), 0, cost.data_ptr(), iters[0].data_ptr(), iters[1].data_ptr(), st.data_ptr())

        def perturbed():
            mpc.closed_loop_perturbed_dev(S, N, K_SIM, I_SIM, EPS, prof, 0, x.data_ptr(), p.data_ptr(), S, pp.data_ptr(), S,
                                          rk4, d.data_ptr(), v.data_ptr(), xk.data_ptr(), uk.data_ptr(), 0,
                                          cost.data_ptr(), iters[0].data_ptr(), iters[1].data_ptr(), st.data_ptr())

        def step_api():
            state.zero_()
            xs[0].copy_(x)
            for k in range(K_SIM):
                a, b = xs[k % 2], xs[(k + 1) % 2]
                torch.add(a, v[:, k], out=y)
                mpc.mpc_step_dev(S, N, I_SIM, EPS, prof, 0, y.data_ptr(), p.data_ptr(), S, state.data_ptr(), u.data_ptr(),
                                 0, sit[0].data_ptr(), sit[1].data_ptr(), sit[2].data_ptr())
                mpc.plant_step_dev(S, rk4, 0, a.data_ptr(), u.data_ptr(), pp.data_ptr(), S, b.data_ptr())
                b.add_(d[:, k])

        arms = dict(fused=lambda: loop(prof), fused_rk4=lambda: loop(prof | rk4), perturbed=perturbed, step_api=step_api)

        def timed(fn):
            e0 = ev()
            fn()
            e1 = ev()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1)

        for fn in arms.values():                                  # warm-up: module load, scratch allocation, caches
            timed(fn)
        ts = {k: [] for k in arms}
        for _ in range(args.repeats):
            for k, fn in arms.items():
                ts[k].append(timed(fn))
        perturbed(); step_api()
        torch.cuda.synchronize()
        same = bool(torch.equal(xs[K_SIM % 2], xk[:, K_SIM, :]))   # c and d end on the same bits

        def rate(t):
            return dict(ms_median=statistics.median(t), ms_min=min(t), ms_max=max(t), ms_all=t,
                        scenario_steps_per_s=S * K_SIM / (statistics.median(t) * 1e-3))

        row = dict(config=cfg, S=S, N=N, **{k: rate(t) for k, t in ts.items()},
                   perturbed_over_fused_rk4=statistics.median(ts["perturbed"]) / statistics.median(ts["fused_rk4"]),
                   step_api_over_perturbed=statistics.median(ts["step_api"]) / statistics.median(ts["perturbed"]),
                   final_state_equals_step_api=same)
        res["configs"].append(row)
        print(json.dumps(dict((k, row[k]) for k in ("config", "S", "N", "perturbed_over_fused_rk4",
                                                    "step_api_over_perturbed", "final_state_equals_step_api")))
              + " " + " ".join(f"{k} {row[k]['ms_median']:.3f} ms" for k in arms), flush=True)
        del p, pp, x, d, v, xk, uk, cost, iters, st, state, xs, y, u, sit
        torch.cuda.empty_cache()
    mpc.reset_stream()
    mpc.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_perturbed.json"), "w") as f:
        json.dump(res, f, indent=1)
    print("device:", res["device"], res["nvidia_smi"])


if __name__ == "__main__":
    main()
