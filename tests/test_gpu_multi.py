"""Multi-GPU behind the drop-in boundary (VERDICT r1 item 4): `ntm_mpc_closed_loop_multi` drives every visible GPU
from ONE host process (what the MEX gateway `ntm_mpc_batch` can reach), and `ntm_mpc_closed_loop_rec_dev` writes the
packed per-scenario record a multi-process caller gathers with a single collective.  Scenarios never interact
(NTM_MPC_Sim.m:93-131), so every sharded result must equal the single-device result BIT FOR BIT.

With one visible GPU the multi entry is exercised with n_devices = 1 and by listing device 0 explicitly; the
>1-device cases skip (they run under `gpurun --gpus 2`, see profiles/)."""
import ctypes
import os

import numpy as np
import pytest

from oracle import ntm_oracle as o

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mpc():
    import ntm_mpc
    h = ntm_mpc.NtmMpc(0)
    yield h
    h.close()


def _same(a, b):
    for k in ("xk", "uk", "cost", "inner_iters", "qp_iters", "status"):
        assert np.array_equal(a[k], b[k], equal_nan=(a[k].dtype.kind == "f")), k


def test_record_entry_equals_the_three_array_entry(mpc):
    import torch
    import ntm_mpc
    from ntm_mpc import physics
    P, x0, N = physics.batch_params(3, S=777)
    prm = np.ascontiguousarray(P.T)
    K = 20
    ref = mpc.closed_loop(x0, prm, N, K, 10, 1e-14, ntm_mpc.PROFILE_INNER_FIXED)
    dev = torch.device("cuda:0")
    d_x0, d_p = torch.from_numpy(x0).to(dev), torch.from_numpy(prm).to(dev)
    ld = ntm_mpc.rec_doubles(K)
    assert ld == 64
    rec = torch.full((777, ld), -7.0, dtype=torch.float64, device=dev)
    inner = torch.zeros((777, K), dtype=torch.int32, device=dev)
    mpc.set_stream(torch.cuda.current_stream(dev).cuda_stream or None)
    try:
        mpc.closed_loop_rec_dev(777, N, K, 10, 1e-14, ntm_mpc.PROFILE_INNER_FIXED, d_x0.data_ptr(), d_p.data_ptr(), 777,
                                rec.data_ptr(), inner.data_ptr(), 0)
        torch.cuda.synchronize()
    finally:
        mpc.reset_stream()
    r = rec.cpu().numpy()
    assert np.array_equal(r[:, :2 * (K + 1)].reshape(777, K + 1, 2), ref["xk"])
    assert np.array_equal(r[:, 2 * (K + 1):3 * K + 2], ref["uk"])
    assert np.array_equal(r[:, 3 * K + 2], ref["cost"])
    assert np.array_equal(r[:, 3 * K + 3].astype(np.int32), ref["status"])
    assert np.array_equal(inner.cpu().numpy(), ref["inner_iters"])


@pytest.mark.parametrize("S", [1, 5, 1000])
def test_multi_entry_on_the_visible_devices_is_bit_identical(mpc, S):
    import ntm_mpc
    from ntm_mpc import physics
    P, x0, N = physics.batch_params(4, S=S)
    prm = np.ascontiguousarray(P.T)
    ref = mpc.closed_loop(x0, prm, N, 20, 10, 1e-14, 0, want_Uk=True)
    nd = ntm_mpc.device_count()
    assert nd >= 1
    for devices in ([0], None, 1):
        got = ntm_mpc.closed_loop_multi(x0, prm, N, 20, 10, 1e-14, 0, want_Uk=True, devices=devices)
        _same(got, ref)
        assert np.array_equal(got["Uk"], ref["Uk"])
    # one shared parameter block, state rows kept
    got = ntm_mpc.closed_loop_multi(x0, prm[0], N, 8, 4, 1e-14, ntm_mpc.PROFILE_INNER_FIXED, state_rows=ntm_mpc.STATE_ROWS_REFRESH)
    ref2 = mpc.closed_loop(x0, prm[0], N, 8, 4, 1e-14, ntm_mpc.PROFILE_INNER_FIXED, state_rows=ntm_mpc.STATE_ROWS_REFRESH)
    _same(got, ref2)


def test_multi_entry_soa_layout_and_argument_errors(mpc):
    """SoA layout (scenario fastest): a shard is a column band of every array (2-D copies)."""
    import ntm_mpc
    from ntm_mpc import _lib, physics
    lib = _lib.load()
    S, K = 300, 6
    P, x0, N = physics.batch_params(3, S=S)                          # P is [16, S] = SoA already
    ref = mpc.closed_loop(x0, np.ascontiguousarray(P.T), N, K, 10, 1e-14, ntm_mpc.PROFILE_INNER_FIXED)
    x0s = np.ascontiguousarray(x0.T)
    xk = np.empty((2 * (K + 1), S)); uk = np.empty((K, S)); cost = np.empty(S)
    inner = np.empty((K, S), dtype=np.int32); qp = np.empty((K, S), dtype=np.int32); st = np.empty(S, dtype=np.int32)
    nd = ntm_mpc.device_count()
    rc = lib.ntm_mpc_closed_loop_multi(0, None, ntm_mpc.LAYOUT_SOA, ntm_mpc.PROFILE_INNER_FIXED, S, N, K, 10, 1e-14, x0s.ctypes.data,
                                       P.ctypes.data, S, 0, None, xk.ctypes.data, uk.ctypes.data, None, cost.ctypes.data,
                                       inner.ctypes.data, qp.ctypes.data, st.ctypes.data)
    assert rc == 0, lib.ntm_last_error()
    assert np.array_equal(xk.T.reshape(S, K + 1, 2), ref["xk"]) and np.array_equal(uk.T, ref["uk"])
    assert np.array_equal(cost, ref["cost"]) and np.array_equal(inner.T, ref["inner_iters"]) and np.array_equal(st, ref["status"])
    bad = (ctypes.c_int * 2)(0, 0)
    assert lib.ntm_mpc_closed_loop_multi(2, bad, 0, 0, S, N, K, 10, 1e-14, x0s.ctypes.data, P.ctypes.data, S, 0, None, xk.ctypes.data,
                                         uk.ctypes.data, None, None, None, None, None) == 1           # listed twice / out of range
    assert lib.ntm_mpc_closed_loop_multi(nd + 1, None, 0, 0, S, N, K, 10, 1e-14, x0s.ctypes.data, P.ctypes.data, S, 0, None,
                                         xk.ctypes.data, uk.ctypes.data, None, None, None, None, None) == 1
    assert lib.ntm_mpc_closed_loop_multi(1, None, 0, 0, S, N, K, 10, 1e-14, x0s.ctypes.data, P.ctypes.data, 7, 0, None,
                                         xk.ctypes.data, uk.ctypes.data, None, None, None, None, None) == 1  # params_count


def test_out_buffers_are_validated(mpc):
    import ntm_mpc
    from ntm_mpc import physics
    P, x0, N = physics.batch_params(3, S=16)
    prm = np.ascontiguousarray(P.T)
    with pytest.raises(ValueError, match="dtype"):
        mpc.closed_loop(x0, prm, N, out=dict(uk=np.empty((16, 20), dtype=np.float32)))
    with pytest.raises(ValueError, match="shape"):
        mpc.closed_loop(x0, prm, N, out=dict(xk=np.empty((16, 20, 2))))
    with pytest.raises(ValueError, match="contiguous"):
        mpc.closed_loop(x0, prm, N, out=dict(uk=np.empty((20, 16)).T))
    with pytest.raises(ValueError, match="dtype"):
        mpc.closed_loop(x0, prm, N, out=dict(status=np.empty(16, dtype=np.int64)))


def test_all_devices_give_the_single_device_result(mpc):
    """> 1 visible GPU: every device count from 2 to all, ragged shards included."""
    import ntm_mpc
    from ntm_mpc import physics
    nd = ntm_mpc.device_count()
    if nd < 2:
        pytest.skip("one visible GPU")
    S = 4099
    P, x0, N = physics.batch_params(3, S=S)
    prm = np.ascontiguousarray(P.T)
    ref = mpc.closed_loop(x0, prm, N, 20, 10, 1e-14, 0)
    for n in range(2, nd + 1):
        _same(ntm_mpc.closed_loop_multi(x0, prm, N, 20, 10, 1e-14, 0, devices=n), ref)
    _same(ntm_mpc.closed_loop_multi(x0, prm, N, 20, 10, 1e-14, 0, devices=[nd - 1, 0]), ref)


def test_mex_batch_gateway_uses_every_gpu():
    """MEX id 8 (`ntm_mpc_batch`) shards over the visible GPUs through ntm_mpc_closed_loop_multi."""
    import ntm_mpc
    from ntm_mpc import physics
    from test_mex_gateway import Mock
    nd = ntm_mpc.device_count()
    if nd < 2:
        pytest.skip("one visible GPU")
    mock = Mock()
    S = 256
    P, x0, N = physics.batch_params(3, S=S)
    os.environ["NTM_MEX_MIN_SHARD"] = "16"                             # 256 / 16 >= nd: all devices take a shard
    try:
        xk, uk, cost, inner, status = mock.call("ntm_mpc_batch", [x0.T, P, N, 20, 10, 1e-14, 16], nlhs=5)
    finally:
        os.environ.pop("NTM_MEX_MIN_SHARD", None)
    h = ntm_mpc.NtmMpc(0)
    ref = h.closed_loop(x0, np.ascontiguousarray(P.T), N, 20, 10, 1e-14, 16)
    h.close()
    assert np.array_equal(uk.T, ref["uk"]) and np.array_equal(xk.T.reshape(S, 21, 2), ref["xk"])
    assert np.array_equal(cost[0], ref["cost"]) and not status.any()
    # the pooled handles of the other devices have launched kernels
    from ntm_mpc import _lib
    assert _lib.load().ntm_pool_launch_count(nd - 1) > 0
