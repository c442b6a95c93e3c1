#!/usr/bin/env python
"""bench.py -- closed-loop LPV-MPC scenario-steps/s on N x B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port; MATLAB absent)
    python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs as DIR/<name>.npy

One *step* = one pass of the hot path over one batch: the whole closed loop NTM_MPC_Sim.m:63-131
(k_sim = 20 MPC steps, i_sim = 10 re-linearisations each under the default `fixed` inner policy) for
every scenario of the batch, in ONE launch of the fused persistent kernel per GPU.

Workloads are the BASELINE.json configs at their STATED TOTAL sizes: config2 = 1,024 scenarios (N = 10),
config3 = 65,536 (N = 20, sampled coefficients; the default -- the configuration the north-star target is quoted
on), config4 = 1,048,576 (N = 20, P_EC boxes that bind), config5 = 16,384 (N = 100).  `--gpus N` SPLITS the named
batch into contiguous shards of ceil(S/N) scenarios (`--scaling strong`, the default: config 3 is "65,536 scenarios
sharded across 8 x B200"); `--scaling weak` gives every rank its own full-size batch instead.  For N > 1 the step
ends with the ONE NCCL all-gather of the packed per-scenario records [xk | uk | cost | status] (64 doubles at
k_sim = 20) that the kernel writes directly (ntm_mpc_closed_loop_rec_dev).

`value`   : scenario-steps/s, inputs resident in HBM, device-timed (CUDA events per step, max over ranks), gather included.
`e2e`     : same metric through the public host API (ntm_mpc.NtmMpc.closed_loop -> C ABI with HOST buffers):
            pinned H2D of x0 + params, kernel, D2H of xk/uk/cost/iters/status every step; `e2e.pageable` is the
            same call on plain NumPy (pageable) buffers -- what a MEX gateway hands over.
`roofline`: the fused kernel is FP64-pipe bound (48 B of mandatory HBM traffic per scenario-step against
            ~1e5 flops): achieved = algorithmic flops (SURVEY 8d formula, QP flops from the kernel's own
            iteration counters) / launch time; peak = DFMA rate measured live by ntm_fp64_peak
            (MEASURED_PEAKS.json carries no FP64 figure).  `roofline_condense` is the HBM-bound
            materialising kernel ntm_condense against MEASURED_PEAKS.json's hbm_gbs.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "mpc-ntm-control_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

K_SIM, I_SIM, EPS = 20, 10, 1e-14
WORKLOADS = {  # name -> (BASELINE config id, TOTAL scenarios of the config as BASELINE.json states it)
    "config2": (2, 1024), "config3": (3, 65536), "config4": (4, 1048576), "config5": (5, 16384),
}
HORIZON = {2: 10, 3: 20, 4: 20, 5: 100}
DUMP_BYTES = 63_000_000      # --dump-outputs stays below 64 MB with the .npy headers; larger batches are sampled


def host_threads() -> int:
    """Host cores this process may use.  NOT omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1 to every
    rank, which silently turned the CPU arm into a 1-core run in round 1."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def flops_per_inner(N: int) -> float:
    """SURVEY 8(d): algorithmic flops of one re-linearisation, QP excluded (dense 2x2 blocks, block-
    triangular zeros skipped, G lower triangle only): 299 / 2385 / 10890 / 778530 at N = 3/10/20/100."""
    g_struct = 3 * N * (N + 1) + (2.0 / 3.0) * N * (N + 1) * (N + 2) + N * (N + 1) / 2.0
    return (14 * N + 4 * N + 12 * (N - 1) + 3 * N * (N - 1) + 8 * (N - 1) + (16 * N + 2 * N * (N + 1) + N)
            + 10 * N + g_struct)


def flops_per_qp_iter(N: int) -> float:
    """one pivoting iteration = one G mat-vec (2N^2) (+ the free-block solve, not counted)."""
    return 2.0 * N * N


def loop_flops(N: int, inner_sum: int, qp_sum: int, scen_steps: int) -> float:
    return inner_sum * flops_per_inner(N) + qp_sum * flops_per_qp_iter(N) + 30.0 * scen_steps


def hess_traffic(S: int, N: int):
    """dram bytes per launch of hessian_grad_dmma_kernel from its committed ncu capture (profiles/traffic.json), only for the
    shape it was captured on."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["hessian_grad_dmma_kernel"]
        return t["dram_bytes_per_launch"] if (t["scenarios"], t["horizon_N"]) == (S, N) else None
    except Exception:
        return None


def ncu_traffic(workload: str, S: int):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the fused kernel from the committed ncu capture
    (profiles/traffic.json); only valid for the shape it was captured on, otherwise null."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["closed_loop_kernel"]
        return int(t["dram_bytes_per_launch"]) if (workload == "config3" and S == 65536) else None
    except Exception:
        return None


def ncu_units():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["closed_loop_kernel"].get("units")
    except Exception:
        return None


def pct(xs, q):
    """q-quantile (nearest rank) of a list."""
    ys = sorted(xs)
    return ys[min(len(ys) - 1, max(0, int(round(q * (len(ys) - 1)))))]


def dump_outputs(path: str, rec: np.ndarray, inner: np.ndarray, qp: np.ndarray) -> None:
    """--dump-outputs: what the timed path returned in its last step, one <path>/<name>.npy per array, scenario-major.
    The packed record [xk | uk | cost | status] is split into xk [S, K+1, 2], uk [S, K], cost [S] and status [S]
    (float64, as the kernel stores them); inner_iters and qp_iters [S, K] are float32 (exact for these counts);
    scenario [S] is each row's index in the batch.  A batch larger than DUMP_BYTES is written as a fixed seeded sample
    of its scenarios, in index order, so that two builds can be compared row for row."""
    S, K = inner.shape
    idx = np.arange(S)
    per_scenario = 8 * rec.shape[1] + 2 * 4 * K + 8
    if S * per_scenario > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(S, DUMP_BYTES // per_scenario, replace=False))
    rec = rec[idx]
    arrays = dict(xk=rec[:, :2 * (K + 1)].reshape(-1, K + 1, 2), uk=rec[:, 2 * (K + 1):3 * K + 2], cost=rec[:, 3 * K + 2],
                  status=rec[:, 3 * K + 3], inner_iters=inner[idx].astype(np.float32), qp_iters=qp[idx].astype(np.float32),
                  scenario=idx.astype(np.float64))
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu: int):
        super().__init__(daemon=True)
        self.gpu, self.rows, self._stop_evt = gpu, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        sm = [float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(self.rows))


def cpu_baseline(config: int, policy_flags: int, target_s: float = 12.0, threads: int = 0, extras: bool = False):
    """The oracle's C restatement (kind 'port': the reference is MATLAB and neither MATLAB nor Octave exists on
    the box) timed on the host cores over a bounded prefix of the same workload."""
    from oracle import c_oracle, ntm_oracle as o
    c_oracle.build()
    threads = threads if threads > 0 else host_threads()
    pilot_S = 64 if config != 5 else 8
    phys, x0, N = o.make_batch(config, S=pilot_S)
    t0 = time.perf_counter()
    r = c_oracle.closed_loop_batch(phys, x0, N, K_SIM, I_SIM, EPS, policy_flags, threads)
    dt = max(time.perf_counter() - t0, 1e-4)
    S = int(min(max(pilot_S, pilot_S * target_s / dt), WORKLOADS.get(f"config{config}", (config, 65536))[1]))
    phys, x0, N = o.make_batch(config, S=S)
    t0 = time.perf_counter()
    r = c_oracle.closed_loop_batch(phys, x0, N, K_SIM, I_SIM, EPS, policy_flags, threads)
    dt = time.perf_counter() - t0
    cores = int(r["threads"])
    if host_threads() > 1 and cores <= 1:
        raise RuntimeError(f"cpu_baseline ran on {cores} core of {host_threads()}: OpenMP team was not honoured")
    out = dict(value=S * K_SIM / dt, unit="scenario-steps/s", cores=cores, kind="port",
               sample=f"first {S} scenarios of config{config} (N={N}, k_sim={K_SIM}), C restatement oracle/ntm_oracle.c, "
                      f"{cores} OpenMP threads, {dt:.2f} s", seconds=dt, scenarios=S, same_config=(S == WORKLOADS[f"config{config}"][1]),
               note="bounded PREFIX of the workload (cost is linear in the scenario count, so the rate carries over)")
    if extras:
        # SURVEY 8(d): the same port on one thread, the NumPy oracle on one core, and the interpreter if one exists
        S1 = max(8, S // (4 * max(cores, 1)))
        ph1, x1, _ = o.make_batch(config, S=S1)
        t0 = time.perf_counter(); c_oracle.closed_loop_batch(ph1, x1, N, K_SIM, I_SIM, EPS, policy_flags, 1); d1 = time.perf_counter() - t0
        Sn = 2
        phn, xn, _ = o.make_batch(config, S=Sn)
        prof = o.LITERAL_FIXED if policy_flags & 16 else o.LITERAL
        t0 = time.perf_counter()
        for s_ in range(Sn):
            o.closed_loop(o.scenario(phn, s_), xn[s_], N=N, profile=prof)
        dn = time.perf_counter() - t0
        import shutil
        interp = shutil.which("matlab") or shutil.which("octave") or shutil.which("octave-cli")
        out["also"] = dict(c_port_1_thread=S1 * K_SIM / d1, numpy_oracle_1_core=Sn * K_SIM / dn,
                           matlab_octave=interp or "unavailable (probed: matlab, octave, octave-cli not on PATH); the committed .m files do not execute either (SURVEY 2.3)")
    return out


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path.  MATLAB/Octave are absent and the
    committed .m files do not execute (SURVEY 2.3), so this is the oracle port on ALL host threads (explicit count:
    torchrun's OMP_NUM_THREADS=1 is ignored)."""
    if rank != 0:
        return
    cfg, S_total = WORKLOADS[args.workload]
    flags = 16 if args.policy == "fixed" else 0
    from oracle import c_oracle, ntm_oracle as o
    c_oracle.build()
    threads = host_threads()
    budget = float(os.environ.get("NTM_BENCH_REF_BUDGET_S", "60"))        # whole-run CPU budget of the reference arm
    pilot = cpu_baseline(cfg, flags, target_s=max(0.2, budget / max(args.steps + args.warmup, 1)), threads=threads)
    S = pilot["scenarios"]
    phys, x0, N = o.make_batch(cfg, S=S)
    times = []
    r = None
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        r = c_oracle.closed_loop_batch(phys, x0, N, K_SIM, I_SIM, EPS, flags, threads)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    cores = int(r["threads"])
    value = S * K_SIM * args.steps / total
    line = dict(metric="closed-loop LPV-MPC scenario-steps/s", value=value, unit="scenario-steps/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * total / args.steps, higher_is_better=True,
                scaling=args.scaling or ("strong" if args.gpus > 1 else "weak"), vs_baseline=None, dtype="f64", data="synthetic",
                impl="reference",
                config=dict(workload=args.workload, scenarios_total=S_total, horizon_N=N, k_sim=K_SIM, i_sim=I_SIM,
                            inner_policy=args.policy, scenarios_per_step=S, same_config=(S == S_total),
                            note="each step = a bounded PREFIX of the workload (first scenarios_per_step scenarios; cost is "
                                 "linear in the scenario count); CPU port of the repaired reference, all host threads"),
                cpu_baseline=dict(value=value, unit="scenario-steps/s", cores=cores, kind="port",
                                  sample=f"first {S} scenarios of {args.workload} per step, {cores} OpenMP threads "
                                         f"(host has {threads})"),
                e2e=dict(value=value, unit="scenario-steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="config3", choices=sorted(WORKLOADS))
    ap.add_argument("--policy", default="fixed", choices=["fixed", "eps_break"])
    ap.add_argument("--scaling", default=None, choices=["strong", "weak"],
                    help="strong (default): --gpus N splits the named config; weak: every rank runs the full-size batch")
    ap.add_argument("--scenarios", type=int, default=0, help="override the TOTAL scenario count of the workload")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary measurements (condense roofline, latency, eps_break)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (native path; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to the native path (the reference arm's batch size depends on its timing)")
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import ntm_mpc
    from ntm_mpc import distributed as D, physics

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    scaling = args.scaling or "strong"
    cfg, S_total = WORKLOADS[args.workload]
    if args.scenarios:
        S_total = args.scenarios
    if scaling == "weak":
        # every rank its own full-size batch (per-rank seeds; rank 0 = the BASELINE batch itself)
        P, x0, N = physics.batch_params(cfg, S=S_total, seed=physics.CONFIG_SHAPES[cfg][0] + rank)
        S = S_total
        S_job = S_total * world
    else:
        # the named batch, cut into contiguous shards of ceil(S/world) scenarios (SURVEY 8e)
        Pf, x0f, N = physics.batch_params(cfg, S=S_total)
        lo, hi = D.shard_range(S_total, world, rank)
        P, x0 = np.ascontiguousarray(Pf[:, lo:hi]), np.ascontiguousarray(x0f[lo:hi])
        S = hi - lo
        S_job = S_total
        del Pf, x0f
    S_pad = D.padded_count(S_total, world) if scaling == "strong" else S       # equal counts for the gather
    flags = ntm_mpc.PROFILE_INNER_FIXED if args.policy == "fixed" else 0

    mpc = ntm_mpc.NtmMpc(local)
    stream = torch.cuda.current_stream()
    mpc.set_stream(stream.cuda_stream)
    fp64_tf, _ = mpc.fp64_peak(1 << 14)
    fp64_tf = max(fp64_tf, mpc.fp64_peak(1 << 14)[0])

    # ---- resident inputs / outputs: ONE packed record per scenario (the block the all-gather moves)
    LD = ntm_mpc.rec_doubles(K_SIM)
    d_x0 = torch.from_numpy(x0).to(dev)
    d_P = torch.from_numpy(np.ascontiguousarray(P.T)).to(dev)
    d_rec = torch.zeros((S_pad, LD), dtype=torch.float64, device=dev)
    d_inner = torch.zeros((max(S, 1), K_SIM), dtype=torch.int32, device=dev)
    d_qp = torch.zeros((max(S, 1), K_SIM), dtype=torch.int32, device=dev)
    g_rec = torch.empty((world * S_pad, LD), dtype=torch.float64, device=dev) if world > 1 else None
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2

    def launch():
        if S > 0:
            mpc.closed_loop_rec_dev(S, N, K_SIM, I_SIM, EPS, flags, d_x0.data_ptr(), d_P.data_ptr(), S, d_rec.data_ptr(),
                                    d_inner.data_ptr(), d_qp.data_ptr())

    def gather():
        if world > 1:                                                # the one collective of the path
            dist.all_gather_into_tensor(g_rec, d_rec)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        launch(); gather()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = mpc.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(args.steps)]
    barrier()
    for e0, ek, e1 in ev:
        flush.zero_()                                                # L2 flush between timed iterations (not timed)
        e0.record(stream)
        launch()
        ek.record(stream)                                            # end of THIS rank's kernel: before the collective
        gather()
        e1.record(stream)
    barrier()
    launches = mpc.launch_count() - launches0
    step_ms = [e0.elapsed_time(e1) for e0, ek, e1 in ev]
    kern_ms = [e0.elapsed_time(ek) for e0, ek, e1 in ev]
    coll_ms = [ek.elapsed_time(e1) for e0, ek, e1 in ev]           # all-gather incl. waiting for the slowest rank
    t3 = torch.tensor([sum(step_ms), sum(kern_ms), -sum(kern_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t3, op=dist.ReduceOp.MAX)
    total_ms, kern_max_ms, kern_min_ms = float(t3[0]), float(t3[1]), -float(t3[2])
    value = S_job * K_SIM * args.steps / (total_ms * 1e-3)

    cnt = torch.tensor([int(d_inner.sum().item()), int(d_qp.sum().item())], dtype=torch.int64, device=dev)
    inner_loc, qp_loc = int(cnt[0]), int(cnt[1])
    if world > 1:
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    inner_sum, qp_sum = int(cnt[0]), int(cnt[1])
    status_max = int(d_rec[:S, 3 * K_SIM + 3].max().item()) if S else 0
    kern_s = statistics.mean(kern_ms) * 1e-3
    flops = loop_flops(N, inner_loc, qp_loc, S * K_SIM)             # this rank's kernel against this rank's GPU
    achieved_tf = flops / kern_s / 1e12 if kern_s > 0 else 0.0
    d_uk_res = d_rec[:S, 2 * (K_SIM + 1):3 * K_SIM + 2].contiguous()
    if args.dump_outputs:
        outs = [d_rec[:S], d_inner[:S], d_qp[:S]]
        if world > 1:                                                # whole job in scenario order, as the gather delivers it
            outs = [D.all_gather_scenarios(t, S_job) for t in outs]
        if rank == 0:
            dump_outputs(args.dump_outputs, *(t.cpu().numpy() for t in outs))

    # ---- e2e: public host API, host buffers, H2D + kernel + D2H every step (pinned, then pageable)
    mpc.reset_stream()
    e2e = {}
    hx_np, hp_np = np.ascontiguousarray(x0), np.ascontiguousarray(P.T)
    parity_probe = None
    for kind in ("pinned", "pageable"):
        if kind == "pinned":
            pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()   # noqa: E731
            hx = torch.from_numpy(hx_np).pin_memory().numpy(); hp = torch.from_numpy(hp_np).pin_memory().numpy()
        else:
            pin = lambda shape, dt: np.empty(shape, dtype=np.float64 if dt == torch.float64 else np.int32)   # noqa: E731
            hx, hp = hx_np.copy(), hp_np.copy()
        out = dict(xk=pin((S, K_SIM + 1, 2), torch.float64), uk=pin((S, K_SIM), torch.float64), cost=pin((S,), torch.float64),
                   inner_iters=pin((S, K_SIM), torch.int32), qp_iters=pin((S, K_SIM), torch.int32), status=pin((S,), torch.int32))
        for _ in range(2):
            if S:
                mpc.closed_loop(hx, hp, N, K_SIM, I_SIM, EPS, flags, out=out)
        barrier()
        n_e2e = args.steps if kind == "pinned" else max(3, min(args.steps, 5))
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            if S:
                mpc.closed_loop(hx, hp, N, K_SIM, I_SIM, EPS, flags, out=out)
        barrier()
        tt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e[kind] = dict(value=S_job * K_SIM * n_e2e / float(tt.item()), steps=n_e2e)
        if kind == "pinned":
            parity_probe = bool(np.array_equal(out["uk"], d_uk_res.cpu().numpy()))      # host path == resident path, bit for bit
    h2d_bytes = S * (2 + ntm_mpc.NPARAM) * 8
    d2h_bytes = S * ((2 * (K_SIM + 1) + K_SIM + 1) * 8 + (2 * K_SIM + 1) * 4)
    clocks = sampler.stop()

    line = dict(metric="closed-loop LPV-MPC scenario-steps/s", value=value, unit="scenario-steps/s", n_gpus=world,
                steps=args.steps, warmup=args.warmup, ms_per_step=total_ms / args.steps, higher_is_better=True,
                scaling=scaling, vs_baseline=None, dtype="f64", data="synthetic",
                config=dict(workload=args.workload, scenarios_total=S_job, scenarios_per_gpu=S, horizon_N=N, k_sim=K_SIM,
                            i_sim=I_SIM, inner_policy=args.policy, profile="literal", parallelism=f"scenario-shard x{world}",
                            l2="flushed between timed steps (256 MiB memset, untimed)",
                            collective=f"ONE all_gather_into_tensor of packed records ({LD} doubles per scenario) inside the step"
                            if world > 1 else "none"),
                e2e=dict(value=e2e["pinned"]["value"], unit="scenario-steps/s", h2d_bytes_per_step=h2d_bytes,
                         d2h_bytes_per_step=d2h_bytes, steps=e2e["pinned"]["steps"], host_buffers="pinned",
                         pageable=dict(value=e2e["pageable"]["value"], steps=e2e["pageable"]["steps"],
                                       note="plain NumPy buffers = what a MEX gateway passes (mxArray memory is pageable)")),
                gpu_launches=int(launches),
                clocks=clocks,
                roofline=dict(bound="fp64", kernel="closed_loop_kernel", achieved=achieved_tf, peak=fp64_tf, unit="TFLOP/s",
                              frac=achieved_tf / fp64_tf if fp64_tf else None, traffic=ncu_traffic(args.workload, S),
                              peak_source="DFMA chain measured live (ntm_fp64_peak); MEASURED_PEAKS.json has no FP64 figure",
                              kernel_ms=statistics.mean(kern_ms), flops_per_launch=flops,
                              launches_per_step=launches / max(args.steps, 1),
                              launch_note="a step of >= 14,800 scenarios is TWO launches of closed_loop_kernel (time step 0, then "
                                          "steps 1..19 in longest-first order) + memset + 3 sort kernels (28 us); kernel_ms and "
                                          "flops_per_launch are per STEP (CUDA events around all of them)",
                              hbm_bytes_per_launch=S * (18 * 8 + LD * 8 + 40 * 4),
                              ncu=ncu_units()),
                counters=dict(mean_inner_iters=inner_sum / max(S_job * K_SIM, 1), mean_qp_iters_per_inner=qp_sum / max(inner_sum, 1),
                              status_max=status_max, host_equals_resident=parity_probe),
                multi_gpu=dict(kernel_ms_max_rank=kern_max_ms / args.steps, kernel_ms_min_rank=kern_min_ms / args.steps,
                               skew_ms=(kern_max_ms - kern_min_ms) / args.steps,
                               allgather_ms=max(0.0, (total_ms - kern_max_ms) / args.steps),
                               collective_incl_wait_ms_this_rank=statistics.mean(coll_ms),
                               gathered_bytes_per_rank=(world * S_pad * LD * 8 if world > 1 else 0)),
                latency=dict(p50_ms_per_launch=pct(kern_ms, 0.5), p99_ms_per_launch=pct(kern_ms, 0.99), launches_timed=len(kern_ms),
                             note=f"one launch = the whole closed loop ({K_SIM} MPC steps) of {S} scenarios on this GPU; "
                                  "per-MPC-step latency of ONE scenario is latency_single below"))

    if rank == 0 and not args.no_extras:
        line.update(extras(mpc, torch, dev, args, ntm_mpc, physics))
    if rank == 0 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(cfg, 16 if args.policy == "fixed" else 0, extras=not args.no_extras)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line), flush=True)


def extras(mpc, torch, dev, args, ntm_mpc, physics):
    """Secondary measurements on rank 0: HBM roofline of the materialising condensation kernel, the tensor-core
    Hessian contraction, every other BASELINE config at its stated size, config 1 and single-step latency."""
    out = {}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    stream = torch.cuda.current_stream()
    mpc.set_stream(stream.cuda_stream)

    def timed(fn, reps=5, flush=None):
        fn(); torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            if flush is not None:
                flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream); fn(); e1.record(stream); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return statistics.median(ts)

    peak64 = max(mpc.fp64_peak(1 << 14)[0], mpc.fp64_peak(1 << 14)[0])
    peak_dmma = max(mpc.dmma_peak(1 << 12)[0], mpc.dmma_peak(1 << 12)[0])

    # (i) ntm_condense, N = 20, 262,144 scenarios: 7,840 B algorithmic per scenario (480 in, 7,360 out) -> 2.06 GB
    S, N = 262144, 20
    rho = torch.rand((3, S, N), dtype=torch.float64, device=dev) * 1e-3 + 1e-3
    prm = torch.from_numpy(physics.params_from_physics(physics.nominal())).to(dev)
    phi = torch.empty(S * 4 * N, dtype=torch.float64, device=dev); gam = torch.empty(S * 2 * N * N, dtype=torch.float64, device=dev)
    lam = torch.empty(S * 2 * N, dtype=torch.float64, device=dev)
    ms = timed(lambda: mpc.condense_dev(S, N, 0, ntm_mpc.LAYOUT_MATLAB, rho[0].data_ptr(), rho[1].data_ptr(), rho[2].data_ptr(),
                                        prm.data_ptr(), 1, phi.data_ptr(), gam.data_ptr(), lam.data_ptr()))
    bytes_alg = S * 8 * (3 * N + 4 * N + 2 * N * N + 2 * N)
    gbs = bytes_alg / (ms * 1e-3) / 1e9
    out["roofline_condense"] = dict(bound="hbm", kernel="condense_kernel", achieved=gbs, peak=hbm_peak, unit="GB/s", frac=gbs / hbm_peak,
                                    traffic=None, peak_source="MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                                    kernel_ms=ms, bytes_per_launch=bytes_alg, scenarios=S, horizon_N=N)
    del rho, phi, gam, lam

    # (i') ntm_hessian_grad at N = 100, 16,384 scenarios (BASELINE config 5's dense Gamma'QGamma contraction) on the
    #      FP64 tensor cores (DMMA.8x8x4).  `achieved`/`frac` count the tensor-core flops actually ISSUED (lower-triangle
    #      tiles only) against the DMMA peak measured live; the dense count 4N^3 + 6N^2 is kept as a note.
    S5, N5 = 16384, 100
    lib = ntm_mpc._lib.load()
    Gam5 = torch.rand((S5, N5, 2 * N5), dtype=torch.float64, device=dev); Phi5 = torch.rand((S5, 2, 2 * N5), dtype=torch.float64, device=dev)
    Lam5 = torch.rand((S5, 2 * N5), dtype=torch.float64, device=dev); x5 = torch.rand((S5, 2), dtype=torch.float64, device=dev)
    G5 = torch.empty((S5, N5, N5), dtype=torch.float64, device=dev); F5 = torch.empty((S5, N5), dtype=torch.float64, device=dev)
    ms = timed(lambda: ntm_mpc._lib.check(lib.ntm_hessian_grad_dev(mpc._h, ntm_mpc.LAYOUT_MATLAB, S5, N5, Phi5.data_ptr(), Gam5.data_ptr(),
                                                                  Lam5.data_ptr(), x5.data_ptr(), prm.data_ptr(), 1, G5.data_ptr(), F5.data_ptr())), reps=3)
    fl_dense = S5 * (4.0 * N5 ** 3 + 6.0 * N5 ** 2)              # dense-no-Omega count of SURVEY 8(a9): both triangles
    nt5 = (N5 + 1 + 7) // 8                                      # tile rows incl. the F row riding along as column N
    fl_exec = S5 * 512.0 * (nt5 * (nt5 + 1) // 2) * ((2 * N5 + 3) // 4)      # DMMA.8x8x4 actually issued
    tf_exec = fl_exec / (ms * 1e-3) / 1e12
    out["roofline_hessian_dmma"] = dict(bound="fp64-tensor", kernel="hessian_grad_dmma_kernel", achieved=tf_exec, peak=peak_dmma,
                                        unit="TFLOP/s", frac=tf_exec / peak_dmma, traffic=hess_traffic(S5, N5), kernel_ms=ms,
                                        flops_per_launch=fl_exec, scenarios=S5, horizon_N=N5,
                                        peak_source="mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4) chains measured live by ntm_dmma_peak",
                                        dense_count=dict(flops=fl_dense, tflops=fl_dense / (ms * 1e-3) / 1e12, dfma_peak=peak64,
                                                         note="4N^3+6N^2 per scenario counts BOTH triangles of the symmetric G; "
                                                              "the kernel computes one -- not a roofline fraction"))
    del Gam5, Phi5, Lam5, x5, G5, F5

    # (ii) every other BASELINE workload at its STATED size (one GPU), both inner policies for the N = 20 configs
    others = []
    for wl, policy in (("config3", "fixed"), ("config3", "eps_break"), ("config2", "fixed"), ("config4", "fixed"),
                       ("config4", "eps_break"), ("config5", "fixed")):
        if wl == args.workload and policy == args.policy:
            continue
        cfg, Sg = WORKLOADS[wl]
        P, x0, Nw = physics.batch_params(cfg, S=Sg)
        fl = ntm_mpc.PROFILE_INNER_FIXED if policy == "fixed" else 0
        dx = torch.from_numpy(x0).to(dev); dP = torch.from_numpy(np.ascontiguousarray(P.T)).to(dev)
        xk = torch.empty((Sg, K_SIM + 1, 2), dtype=torch.float64, device=dev); uk = torch.empty((Sg, K_SIM), dtype=torch.float64, device=dev)
        inn = torch.empty((Sg, K_SIM), dtype=torch.int32, device=dev); qp = torch.empty((Sg, K_SIM), dtype=torch.int32, device=dev)
        st = torch.empty((Sg,), dtype=torch.int32, device=dev)
        ms = timed(lambda: mpc.closed_loop_dev(Sg, Nw, K_SIM, I_SIM, EPS, fl, ntm_mpc.LAYOUT_MATLAB, dx.data_ptr(), dP.data_ptr(), Sg,
                                               xk.data_ptr(), uk.data_ptr(), 0, 0, inn.data_ptr(), qp.data_ptr(), st.data_ptr()),
                   reps=1 if wl == "config5" else 3)
        isum, qsum = int(inn.sum().item()), int(qp.sum().item())
        umax = dP[:, 9:10]
        tf = loop_flops(Nw, isum, qsum, Sg * K_SIM) / (ms * 1e-3) / 1e12
        others.append(dict(workload=wl, scenarios=Sg, horizon_N=Nw, inner_policy=policy, ms=ms,
                           scenario_steps_per_s=Sg * K_SIM / (ms * 1e-3), mean_inner_iters=isum / (Sg * K_SIM),
                           mean_qp_iters_per_inner=qsum / max(isum, 1), status_max=int(st.max().item()),
                           roofline_frac=tf / peak64, achieved_tflops=tf,
                           inner_iters_hist=torch.bincount(inn.flatten().long(), minlength=I_SIM + 1)[1:].tolist(),
                           active_bound_fraction=float(((uk == 0) | (uk == umax)).double().mean().item())))
        others[-1]["profile"] = "literal"
        if wl == "config5":
            others[-1]["note"] = ("literal reading only: the consistent profile at N = 100 is not parity-tested (about 97 % of its "
                                  "scenarios are bit-chaotic in fp64, DESIGN.md section 2); parity of this line: 256 scenarios vs the C oracle")
        del dx, dP, xk, uk, inn, qp, st
    out["other_workloads"] = others

    # (ii') the "next" rows of SURVEY 8(f) inside the same fused loop, config 3 at its stated size: RK4 plant, tau_E(w)
    #       hook, and the QP of NTM_MPC_Sim.m:97 with getWLc's state rows kept (refreshed / frozen, script box :39-45)
    cfg, Sg = WORKLOADS["config3"]
    P, x0, Nw = physics.batch_params(cfg, S=Sg, sample={"c_tauE": (0.3, 1.5)})
    dx = torch.from_numpy(x0).to(dev); dP = torch.from_numpy(np.ascontiguousarray(P.T)).to(dev)
    xk = torch.empty((Sg, K_SIM + 1, 2), dtype=torch.float64, device=dev); uk = torch.empty((Sg, K_SIM), dtype=torch.float64, device=dev)
    inn = torch.empty((Sg, K_SIM), dtype=torch.int32, device=dev); qp = torch.empty((Sg, K_SIM), dtype=torch.int32, device=dev)
    st = torch.empty((Sg,), dtype=torch.int32, device=dev)
    script_box = (0.06, 0.15, 200 * math.pi, 10000 * math.pi)
    FX = ntm_mpc.PROFILE_INNER_FIXED
    nxt = []
    for name, prof, rows in (("rk4_plant", FX | ntm_mpc.PROFILE_PLANT_RK4, 0), ("tau_E_of_w", FX | ntm_mpc.PROFILE_TAUE_W, 0),
                             ("state_rows_refresh_script_box", FX, ntm_mpc.STATE_ROWS_REFRESH),
                             ("state_rows_frozen_script_box", FX, ntm_mpc.STATE_ROWS_FROZEN)):
        if rows:
            fn = lambda: mpc.closed_loop_sc_dev(Sg, Nw, K_SIM, I_SIM, EPS, prof, ntm_mpc.LAYOUT_MATLAB, dx.data_ptr(), dP.data_ptr(), Sg,
                                                rows, script_box, xk.data_ptr(), uk.data_ptr(), 0, 0, inn.data_ptr(), qp.data_ptr(), st.data_ptr())
        else:
            fn = lambda: mpc.closed_loop_dev(Sg, Nw, K_SIM, I_SIM, EPS, prof, ntm_mpc.LAYOUT_MATLAB, dx.data_ptr(), dP.data_ptr(), Sg,
                                             xk.data_ptr(), uk.data_ptr(), 0, 0, inn.data_ptr(), qp.data_ptr(), st.data_ptr())
        ms = timed(fn, reps=2)
        stv = st.cpu().numpy()
        executed = float((inn > 0).sum().item())
        nxt.append(dict(option=name, workload="config3", scenarios=Sg, horizon_N=Nw, inner_policy="fixed", ms=ms,
                        scenario_steps_per_s_nominal=Sg * K_SIM / (ms * 1e-3), scenario_steps_per_s_executed=executed / (ms * 1e-3),
                        mean_qp_iters_per_inner=float(qp.double().sum().item()) / max(float(inn.double().sum().item()), 1.0),
                        status_counts=dict(ok=int((stv == 0).sum()), iter_cap=int((stv == 1).sum()), nonfinite=int((stv == 2).sum()),
                                           infeasible=int((stv == 3).sum()))))
    out["next_rows"] = dict(note="SURVEY 8(f) options in the fused loop; an infeasible QP (quadprog exitflag -2, NTM_MPC_Sim.m:100-101) ends "
                                 "its scenario, so 'executed' counts the scenario-steps that really ran", runs=nxt)
    del dx, dP, xk, uk, inn, qp, st

    # (iii) config 1: the script's own default scenario (S = 1, N = 3) through the HOST API, next to the CPU port
    P1 = physics.params_from_physics(physics.nominal()); x1 = physics.x0_default()
    mpc.reset_stream()
    lat1 = []
    for i in range(40):
        t0 = time.perf_counter()
        r1 = mpc.closed_loop(x1, P1, N=3, k_sim=K_SIM, i_sim=I_SIM, eps=EPS, profile=ntm_mpc.PROFILE_INNER_FIXED)
        if i >= 8:
            lat1.append((time.perf_counter() - t0) * 1e3)
    cfg1 = dict(workload="config1", scenarios=1, horizon_N=3, inner_policy="fixed",
                gpu_ms_e2e_p50=pct(lat1, 0.5), gpu_ms_e2e_p99=pct(lat1, 0.99),
                gpu_scenario_steps_per_s=K_SIM / (pct(lat1, 0.5) * 1e-3), status=int(r1["status"][0]))
    try:
        from oracle import c_oracle, ntm_oracle as o
        c_oracle.build()
        ph, xo, _ = o.make_batch(1)
        tc = []
        for _ in range(20):
            t0 = time.perf_counter(); c_oracle.closed_loop_batch(ph, xo, 3, K_SIM, I_SIM, EPS, 16, 1); tc.append((time.perf_counter() - t0) * 1e3)
        cfg1["cpu_port_ms_p50"] = pct(tc, 0.5)
        cfg1["cpu_port_scenario_steps_per_s"] = K_SIM / (pct(tc, 0.5) * 1e-3)
        cfg1["note"] = "one scenario cannot fill a GPU: launch + PCIe latency dominates; the CPU port wins here by construction"
    except Exception as exc:                                      # the checker is optional for this line
        cfg1["cpu_port_ms_p50"] = None; cfg1["note"] = f"oracle unavailable: {exc}"
    out["config1"] = cfg1
    mpc.set_stream(stream.cuda_stream)

    # (iv) single-scenario single-MPC-step latency through the device-pointer ABI (launch + kernel + sync), N = 20
    P, x0, Nw = physics.batch_params(3, S=1)
    dx = torch.from_numpy(x0).to(dev); dP = torch.from_numpy(np.ascontiguousarray(P.T)).to(dev)
    xk = torch.empty((1, 2, 2), dtype=torch.float64, device=dev); uk = torch.empty((1, 1), dtype=torch.float64, device=dev)
    lat = []
    for i in range(210):
        t0 = time.perf_counter()
        mpc.closed_loop_dev(1, Nw, 1, I_SIM, EPS, ntm_mpc.PROFILE_INNER_FIXED, ntm_mpc.LAYOUT_MATLAB, dx.data_ptr(), dP.data_ptr(), 1,
                            xk.data_ptr(), uk.data_ptr())
        torch.cuda.synchronize()
        if i >= 10:
            lat.append((time.perf_counter() - t0) * 1e6)
    out["latency_single"] = dict(p50_us_one_scenario_one_mpc_step=pct(lat, 0.5), p99_us=pct(lat, 0.99), samples=len(lat),
                                 horizon_N=Nw, i_sim=I_SIM)
    mpc.reset_stream()
    return out


if __name__ == "__main__":
    main()
