"""bench.py contract: the reference arm prints ONE JSON line with the keys a caller reads; --dump-outputs writes what the
timed path returned (-m gpu for the native run)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMPED = ("xk", "uk", "cost", "status", "inner_iters", "qp_iters", "scenario")


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, NTM_BENCH_REF_BUDGET_S="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "scenario-steps/s" and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["dtype"] == "f64" and d["config"]["workload"] == "config3"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_arm_ignores_torchruns_omp_num_threads():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; in round 1 that silently made the CPU arm a 1-core run and
    inflated every N >= 2 speed-up 29x.  The arm must pass its own thread count (host affinity)."""
    ncores = len(os.sched_getaffinity(0))
    if ncores < 2:
        return
    env = dict(os.environ, NTM_BENCH_REF_BUDGET_S="2", OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2", LOCAL_RANK="0")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.strip().startswith("{")][0])
    assert d["cpu_baseline"]["cores"] == ncores, d["cpu_baseline"]
    assert d["n_gpus"] == 2 and d["scaling"] == "strong" and d["config"]["scenarios_total"] == 65536
    # the other ranks exit 0 without work or output
    env["RANK"] = "1"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_native_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


def test_committed_traffic_figures_feed_the_roofline_objects():
    """roofline.traffic / roofline_hessian_dmma.traffic come from the committed ncu captures (profiles/traffic.json) and only
    for the shape they were captured on."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    assert b.hess_traffic(16384, 100) == t["hessian_grad_dmma_kernel"]["dram_bytes_per_launch"] > 3.9e9
    assert b.hess_traffic(8192, 64) is None
    assert b.ncu_traffic("config3", 65536) == t["closed_loop_kernel"]["dram_bytes_per_launch"]
    assert b.ncu_traffic("config3", 8192) is None


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode != 0 and "--steps must be at least 1" in out.stderr


def test_dump_of_a_large_batch_is_a_fixed_sample_below_64_mb(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    S, K = 100_000, 20                                               # 68 MB of outputs in full
    rec = np.repeat(np.arange(S, dtype=np.float64)[:, None], 3 * K + 4, axis=1)
    inner = np.full((S, K), 10, dtype=np.int32)
    qp = np.repeat(np.arange(S, dtype=np.int32)[:, None] % 4096, K, axis=1)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), rec, inner, qp)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64_000_000
    a = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in DUMPED}
    idx = a["scenario"]
    assert 0 < idx.size < S and np.all(np.diff(idx) > 0)
    assert np.array_equal(a["cost"], idx) and np.array_equal(a["xk"][:, 3, 1], idx)    # rows are the sampled scenarios
    assert np.array_equal(a["qp_iters"][:, 0], idx % 4096) and a["xk"].shape == (idx.size, K + 1, 2)
    for n in DUMPED:
        assert a[n].dtype in (np.float32, np.float64), n
        assert np.array_equal(a[n], np.load(tmp_path / "b" / f"{n}.npy")), n     # same sample every time


@pytest.mark.gpu
def test_dump_outputs_are_what_the_timed_path_returns(tmp_path):
    """The native run's dump equals the host API's closed loop on the same seeded batch, bit for bit."""
    import ntm_mpc
    from ntm_mpc import physics
    S = 3000
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--scenarios", str(S),
                          "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = {n: np.load(tmp_path / f"{n}.npy") for n in DUMPED}
    P, x0, N = physics.batch_params(3, S=S)
    mpc = ntm_mpc.NtmMpc(0)
    try:
        ref = mpc.closed_loop(x0, P.T, N=N, profile=ntm_mpc.PROFILE_INNER_FIXED)
    finally:
        mpc.close()
    assert np.array_equal(d["scenario"], np.arange(S))
    for k in DUMPED[:-1]:
        assert d[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(d[k], ref[k]), k
