#!/usr/bin/env python
"""Short horizons (N <= 24, one warp per scenario) of the fused loop against the C oracle: several horizons, both inner
policies, configs 2-4, ragged batch sizes; then config 3 / config 2 / config 4 timings.  GPU box only.
    python tools/check_short.py [quick]"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "mpc-ntm-control_b200")):
    sys.path.insert(0, p)
import numpy as np
import ntm_mpc
from ntm_mpc import physics
from oracle import c_oracle, ntm_oracle as o

mpc = ntm_mpc.NtmMpc(0)
threads = len(os.sched_getaffinity(0))
quick = "quick" in sys.argv


def compare(cfg, S, N, flags=16, k_sim=20, i_sim=10, seed=None):
    phys, x0, _ = o.make_batch(cfg, S=S, seed=seed)
    P = physics.params_from_physics(phys).reshape(16, -1)
    g = mpc.closed_loop(x0, np.ascontiguousarray(P.T), N, k_sim, i_sim, 1e-14, flags, want_Uk=True)
    c = c_oracle.closed_loop_batch(phys, x0, N, k_sim, i_sim, 1e-14, flags & (31 | 64), threads, want_Uk=True)
    umax = np.broadcast_to(np.asarray(phys["umax"], dtype=float), (S,))
    du = np.max(np.abs(g["uk"] - c["uk"]), axis=1) / umax
    dU = np.max(np.abs(g["Uk"] - c["Uk"]).reshape(S, -1), axis=1) / umax
    wref = np.maximum(np.max(np.abs(c["xk"][:, :, 0]), axis=1), 1e-3)
    dw = np.max(np.abs(g["xk"][:, :, 0] - c["xk"][:, :, 0]), axis=1) / wref
    dc = np.max(np.abs(g["cost"] - c["cost"]) / np.maximum(np.abs(c["cost"]), 1e-300))
    bad = (du > 1e-6) | (dw > 1e-6)
    print(f"cfg{cfg} N={N:2d} S={S:4d} k={k_sim:2d} i={i_sim:2d} flags={flags:2d}: du={du.max():.1e} dU={dU.max():.1e} dw={dw.max():.1e} dcost={dc:.1e} "
          f"bad={int(bad.sum())} status {g['status'].max()}/{c['status'].max()} qp/inner {g['qp_iters'].sum() / max(g['inner_iters'].sum(), 1):.3f}/"
          f"{c['qp_iters'].sum() / max(c['inner_iters'].sum(), 1):.3f} inner eq {np.mean(g['inner_iters'] == c['inner_iters']):.4f}"
          + (f"  first bad {int(np.argmax(bad))}" if bad.any() else ""), flush=True)
    return int(bad.sum())


nbad = 0
for N in ([3, 10, 20] if quick else [1, 2, 3, 4, 5, 8, 10, 13, 16, 17, 20, 21, 24]):
    for cfg in (2, 3, 4):
        for flags in (16, 0):
            nbad += compare(cfg, 257 if N >= 8 else 33, N, flags=flags, k_sim=20 if N in (3, 10, 20) else 6)
nbad += compare(3, 4099, 20)
nbad += compare(4, 4099, 20, flags=0)
nbad += compare(3, 1000, 20, flags=16 | 1)            # rho1 squared
nbad += compare(3, 1000, 20, flags=4 | 8)             # F from xk, plant + C (literal Gamma index)
nbad += compare(3, 1000, 20, flags=16 | 64)           # RK4 plant
nbad += compare(1, 1, 3)                              # the script's own scenario
print("total bad", nbad, flush=True)

import torch
dev = torch.device("cuda:0")
stream = torch.cuda.current_stream(); mpc.set_stream(stream.cuda_stream)
for cfg, S, flags in ((3, 65536, 16), (3, 65536, 0), (2, 1024, 16), (4, 1048576, 16), (3, 8192, 16)):
    P, x0, N = physics.batch_params(cfg, S=S)
    dx = torch.from_numpy(x0).to(dev); dP = torch.from_numpy(np.ascontiguousarray(P.T)).to(dev)
    xk = torch.empty((S, 21, 2), dtype=torch.float64, device=dev); uk = torch.empty((S, 20), dtype=torch.float64, device=dev)
    inn = torch.empty((S, 20), dtype=torch.int32, device=dev); qp = torch.empty((S, 20), dtype=torch.int32, device=dev)
    st = torch.empty((S,), dtype=torch.int32, device=dev)
    ts = []
    for rep in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        mpc.closed_loop_dev(S, N, 20, 10, 1e-14, flags, 0, dx.data_ptr(), dP.data_ptr(), S, xk.data_ptr(), uk.data_ptr(), 0, 0,
                            inn.data_ptr(), qp.data_ptr(), st.data_ptr())
        e1.record(stream); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ms = min(ts[1:])
    print(f"config{cfg} S={S} N={N} flags={flags}: {ms:.3f} ms = {S * 20 / ms * 1e3 / 1e6:.2f} M scenario-steps/s, qp/inner {qp.sum().item() / inn.sum().item():.3f}, "
          f"inner/step {inn.sum().item() / (S * 20):.2f}, status max {st.max().item()}, uk sum {float(uk.sum().item()):.17g}", flush=True)
mpc.reset_stream()
