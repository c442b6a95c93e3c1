"""The C ABI's argument contract, entry by entry: a call with one bad argument returns NTM_ERR_INVALID with a message and
leaves no trace -- no launch, no output written and, for a host-pointer entry, no copy in the CUDA activity trace
(include/ntm_mpc.h).  At S == 0 each family of fused entries checks exactly what it documents."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

S, N, K, M = 4, 8, 3, 3                       # scenarios, horizon, k_sim and inequality rows of the valid calls
NMAX = 128                                    # buffers hold the longest horizon a bad call passes
XB = (0.05, 0.16, 2000.0, 12000.0)
XB_INVERTED = (0.16, 0.05, 2000.0, 12000.0)
GAMMA_I, DENSE_G, TAUE_W = 2, 32, 128
SENT = -123
F8, I4 = np.float64, np.int32

# ---------------------------------------------------------------------------------------------- the 14 fused entries
LOOP = ["h", "layout", "profile", "S", "N", "k_sim", "i_sim", "eps", "x0", "params", "pc"]
STEP = ["h", "layout", "profile", "S", "N", "i_sim", "eps", "x0", "params", "pc"]
ROWS = ["state_rows", "xbounds"]
PLANT = ["plant_params", "ppc", "plant_profile", "w", "v"]
OUT = ["xk", "uk", "Uk", "cost", "inner", "qpit", "status"]
FUSED = {"ntm_mpc_closed_loop": LOOP + OUT, "ntm_mpc_closed_loop_sc": LOOP + ROWS + OUT,
         "ntm_mpc_step": STEP + ["state", "uk", "Uk", "inner", "qpit", "status"],
         "ntm_mpc_step_sc": STEP + ROWS + ["state", "uk", "Uk", "inner", "qpit", "status"],
         "ntm_mpc_closed_loop_perturbed": LOOP + PLANT + OUT,
         "ntm_mpc_closed_loop_perturbed_sc": LOOP + ROWS + PLANT + OUT}
FUSED.update({k + "_dev": v for k, v in list(FUSED.items())})
FUSED["ntm_mpc_closed_loop_rec_dev"] = ["h"] + LOOP[2:] + ROWS + ["rec", "inner", "qpit"]
FUSED["ntm_mpc_closed_loop_multi"] = ["n_devices", "devices"] + LOOP[1:] + ROWS + OUT
FUSED_SPEC = {"x0": 2, "params": 16, "plant_params": 16, "w": 2 * K, "v": 2 * K, "xk": 2 * (K + 1), "uk": K,
              "Uk": NMAX * K, "cost": 1, "inner": (K, I4), "qpit": (K, I4), "status": (1, I4), "state": 7 * NMAX + 7,
              "rec": 3 * K + 4}                # elements per scenario

rows = lambda args: "state_rows" in args
controller = lambda args: "state" in args or "plant_profile" in args   # the step's controller (no TAUE_W)
# one bad argument each; a case applies to the entries that take every argument it sets and pass its filter
FUSED_BAD = [
    dict(h=None), dict(layout=7), dict(S=-1), dict(N=0), dict(N=129), dict(k_sim=-1), dict(i_sim=0),
    dict(params=None), dict(pc=3), dict(x0=None), dict(xk=None), dict(uk=None), dict(state=None), dict(rec=None),
    dict(state_rows=3), dict(state_rows=-1), dict(xbounds=None), dict(xbounds=XB_INVERTED),
    dict(xbounds=(np.nan, 0.16, 2000.0, 12000.0)),
    (dict(profile=GAMMA_I, N=40), rows), (dict(profile=DENSE_G, N=33), rows), (dict(N=NMAX), rows),
    (dict(profile=TAUE_W), controller), dict(ppc=3), dict(plant_profile=GAMMA_I),
    dict(devices=[99]), dict(n_devices=2, devices=[0, 0]), dict(n_devices=65),
]


@pytest.fixture(scope="module")
def mpc():
    import ntm_mpc
    h = ntm_mpc.NtmMpc(0)
    yield h
    h.close()


class Entry:
    """One entry point with valid arguments (scalars and buffers on the host or the device, per its flavour); a call
    overrides any of them by name."""

    def __init__(self, mpc, name, args, spec, outputs, scalars, fill):
        import torch
        from ntm_mpc import _lib
        self.lib, self.name, self.args, self.outputs = _lib.load(), name, args, outputs
        self.dev = name.endswith("_dev")
        self.scalars = dict(scalars, h=mpc._h)
        self.bufs = {}
        for k, (count, dtype) in spec.items():
            if k in args:
                a = np.zeros(count, dtype=dtype)
                if k in fill:
                    a[: fill[k].size] = fill[k]
                self.bufs[k] = torch.from_numpy(a).cuda() if self.dev else a
        multi = name.endswith("_multi")
        self.count = (lambda: self.lib.ntm_pool_launch_count(0)) if multi else mpc.launch_count

    def call(self, **over):
        vals = dict(self.scalars, **self.bufs)
        vals.update(over)
        keep = []

        def ptr(v):
            if isinstance(v, (tuple, list)):                 # host arrays in both flavours: xbounds, bounds, devices
                keep.append(np.array(v, dtype=I4 if isinstance(v, list) else F8))
                return keep[-1].ctypes.data
            if isinstance(v, np.ndarray):
                return v.ctypes.data
            return v.data_ptr() if hasattr(v, "data_ptr") else v
        return getattr(self.lib, self.name)(*[ptr(vals[a]) for a in self.args])

    def arm(self):
        """outputs to the sentinel (a controller record is an output too)"""
        for k in self.outputs:
            if self.dev:
                self.bufs[k].fill_(SENT)
            else:
                self.bufs[k].fill(SENT)

    def untouched(self):
        import torch
        if self.dev:
            torch.cuda.synchronize()
        return [k for k in self.outputs if not bool((self.bufs[k] == SENT).all())]

    def valid(self):
        """one valid call: returns the number of kernels it launched"""
        if "state" in self.bufs:
            self.bufs["state"].fill(0)                       # a fresh controller record
        before = self.count()
        assert self.call() == 0, self.lib.ntm_last_error()
        return self.count() - before


def _cuda_activity(fn):
    """(memory copies, kernels) of the CUDA activity trace while fn runs"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return sum(e.name.startswith("Memcpy") for e in ev), sum(not e.name.startswith(("Memcpy", "Memset")) for e in ev)


def reject(e, bad):
    """every call of `bad` returns 1 with a message, launches nothing and writes no output"""
    e.arm()
    for over in bad:
        before = e.count()
        assert e.call(**over) == 1, over
        assert e.lib.ntm_last_error().decode(), over
        assert e.count() == before, over
    assert e.untouched() == [], e.untouched()


def trace(e, bad):
    """The bad calls of a host entry in one profiler window that ends with a valid call, and the same valid call in a
    window of its own: (memory copies, kernels) of both windows and the kernels the valid call counted."""
    e.valid()                                                 # warm-up: module loads, arena, pooled handle
    n = []
    alone = _cuda_activity(lambda: n.append(e.valid()))
    return dict(alone=alone, after_bad=_cuda_activity(lambda: (reject(e, bad), e.valid())), launches=n[0])


def check_trace(t, launches=None):
    """the profiler sees the valid call's copies and launches, and nothing of the bad calls"""
    assert "error" not in t, t
    alone = tuple(t["alone"])
    assert alone[0] >= 2 and alone[1] == t["launches"] >= 1, t
    assert launches is None or t["launches"] == launches, t
    assert tuple(t["after_bad"]) == alone, t


@pytest.fixture(scope="module")
def traces():
    """trace() of every host entry, run once in a child process (python <this file>) so that its profiler sessions
    share no profiler state with the tests of this process"""
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def fused_entry(mpc, name):
    from ntm_mpc import physics
    P, x0, _ = physics.batch_params(3, S=S)
    spec = {k: (v[0] * S, v[1]) if isinstance(v, tuple) else (v * S, F8) for k, v in FUSED_SPEC.items()}
    params = np.ascontiguousarray(P.T).ravel()
    args = FUSED[name]
    outputs = [k for k in OUT + ["state", "rec"] if k in args]
    scalars = dict(layout=0, profile=0, S=S, N=N, k_sim=K, i_sim=3, eps=1e-14, pc=1, ppc=1, plant_profile=0,
                   state_rows=1, xbounds=XB, n_devices=1, devices=None)
    return Entry(mpc, name, args, spec, outputs, scalars,
                 {"x0": np.ascontiguousarray(x0).ravel(), "params": params, "plant_params": params})


def fused_bad(args):
    out = []
    for case in FUSED_BAD:
        over, applies = case if isinstance(case, tuple) else (case, lambda a: True)
        if all(k in args for k in over) and applies(args):
            out.append(over)
    return out


@pytest.mark.parametrize("name", list(FUSED))
def test_fused_entry_rejects_every_bad_argument_without_a_trace(mpc, traces, name):
    e = fused_entry(mpc, name)
    bad = fused_bad(e.args)
    assert len(bad) >= 12, bad
    if not e.dev:
        e.valid()                                             # the pooled handles of _multi exist after a first call
    reject(e, bad)
    if not e.dev:
        check_trace(traces[name], launches=1)


# ---------------------------------------------------------------------------------------------- S == 0, per family
LOOPS = ["ntm_mpc_closed_loop", "ntm_mpc_closed_loop_sc", "ntm_mpc_closed_loop_perturbed",
         "ntm_mpc_closed_loop_perturbed_sc"]
LOOPS += [n + "_dev" for n in LOOPS] + ["ntm_mpc_closed_loop_rec_dev", "ntm_mpc_closed_loop_multi"]
STEPS = ["ntm_mpc_step", "ntm_mpc_step_sc", "ntm_mpc_step_dev", "ntm_mpc_step_sc_dev"]
EVERYTHING_ELSE = dict(N=0, k_sim=-1, i_sim=0, params=None, pc=7, x0=None, xk=None, uk=None, state=None, rec=None,
                       state_rows=7, xbounds=None, profile=TAUE_W, ppc=7, plant_profile=GAMMA_I)
ARRAYS_AND_PARAMS = dict(params=None, pc=7, x0=None, uk=None, state=None)


@pytest.mark.parametrize("name", LOOPS)
def test_a_loop_at_zero_scenarios_checks_only_handle_layout_and_S(mpc, name):
    e = fused_entry(mpc, name)
    other = {k: v for k, v in EVERYTHING_ELSE.items() if k in e.args}
    before = e.count()
    assert e.call(S=0, **other) == 0, e.lib.ntm_last_error()
    assert e.count() == before
    wrong = [dict(layout=7), dict(h=None), dict(devices=[99]), dict(n_devices=2, devices=[0, 0])]
    for over in [w for w in wrong if all(k in e.args for k in w)]:
        assert e.call(S=0, **dict(other, **over)) == 1, over


@pytest.mark.parametrize("name", STEPS)
def test_a_step_at_zero_scenarios_checks_all_but_its_params_and_arrays(mpc, name):
    e = fused_entry(mpc, name)
    before = e.count()
    assert e.call(S=0, **ARRAYS_AND_PARAMS) == 0, e.lib.ntm_last_error()
    bad = [dict(h=None), dict(layout=7), dict(profile=TAUE_W), dict(N=0), dict(N=129), dict(i_sim=0)]
    if "state_rows" in e.args:
        bad += [dict(state_rows=7), dict(xbounds=None), dict(xbounds=XB_INVERTED), dict(profile=GAMMA_I, N=40),
                dict(N=NMAX)]
    for over in bad:
        assert e.call(S=0, **dict(ARRAYS_AND_PARAMS, **over)) == 1, over
    assert e.count() == before


# ---------------------------------------------------------------------------------------------- per-call operations
def _percall_spec():
    n, r = NMAX, 6 * NMAX + 4
    per = {"x": 2, "params": 16, "r1": n, "r2": n, "r3": n, "A": 4, "B": 2, "Phi": 4 * n, "Gamma": 2 * n * n,
           "Lambda": 2 * n, "G": n * n, "F": n, "lb": n, "ub": n, "U": n, "iters": (1, I4), "status": (1, I4),
           "Lg": M * n, "bg": M, "u": 1, "xn": 2, "W": 2 * r, "L": n * r, "c": r, "xk": 2 * (K + 1), "uk": K,
           "cost": 1, "mstatus": (1, I4)}
    spec = {k: (v[0] * S, v[1]) if isinstance(v, tuple) else (v * S, F8) for k, v in per.items()}
    spec["out"] = (22 + 32, F8)
    return spec


PERCALL = {   # name: (arguments, outputs)
    "ntm_rho": (["h", "layout", "profile", "S", "x", "params", "pc", "r1", "r2", "r3"], ["r1", "r2", "r3"]),
    "ntm_lpv_AB": (["h", "layout", "S", "r1", "r2", "r3", "params", "pc", "A", "B"], ["A", "B"]),
    "ntm_condense": (["h", "layout", "profile", "S", "N", "r1", "r2", "r3", "params", "pc", "Phi", "Gamma", "Lambda"],
                     ["Phi", "Gamma", "Lambda"]),
    "ntm_hessian_grad": (["h", "layout", "S", "N", "Phi", "Gamma", "Lambda", "x", "params", "pc", "G", "F"], ["G", "F"]),
    "ntm_qp_box": (["h", "layout", "S", "N", "G", "F", "lb", "ub", "bc", "U", "iters", "status"], ["U", "iters", "status"]),
    "ntm_qp_ineq": (["h", "layout", "S", "N", "M", "G", "F", "lb", "ub", "bc", "Lg", "bg", "U", "iters", "status"],
                    ["U", "iters", "status"]),
    "ntm_plant_step": (["h", "layout", "profile", "S", "x", "u", "params", "pc", "xn"], ["xn"]),
    "ntm_getWLc": (["h", "layout", "S", "N", "bounds", "Gamma", "Phi", "Lambda", "W", "L", "c"], ["W", "L", "c"]),
    "ntm_mc_stats": (["h", "layout", "S", "k_sim", "xk", "uk", "cost", "mstatus", "params", "pc", "bounds", "w_sup",
                      "hist_max", "out"], ["out"]),
}
PERCALL_BAD = [dict(h=None), dict(layout=7), dict(S=-1), dict(N=0), dict(N=129), dict(params=None), dict(pc=3),
               dict(bc=3), dict(M=-1), dict(k_sim=0), dict(bounds=None), dict(out=None),
               dict(N=NMAX, M=1)]                       # ntm_qp_ineq: the factor pair does not fit shared memory


def percall_entry(mpc, name):
    from ntm_mpc import physics
    args, outputs = PERCALL[name.removesuffix("_dev")]
    P, x0, _ = physics.batch_params(3, S=S)
    scalars = dict(layout=0, profile=0, S=S, N=N, M=M, pc=1, bc=S, k_sim=K, w_sup=0.06, hist_max=0.2,
                   bounds=(0.16, 12000.0, 0.05, 2000.0, 2e6, 0.0))
    fill = {"x": np.ascontiguousarray(x0).ravel(), "params": np.ascontiguousarray(P.T).ravel(),
            "G": np.tile(np.eye(N).ravel(), S), "lb": -np.ones(N * S), "ub": np.ones(N * S), "bg": np.full(M * S, 10.0),
            "r1": np.full(N * S, 12.0), "r2": np.full(N * S, 1e-6), "r3": np.full(N * S, 0.03),
            "xk": np.tile([0.08, 6000.0], (K + 1) * S), "uk": np.full(K * S, 1e5)}
    return Entry(mpc, name, args, _percall_spec(), outputs, scalars, fill)


def percall_bad(e):
    ineq = e.name.startswith("ntm_qp_ineq")
    bad = [over for over in PERCALL_BAD if all(k in e.args for k in over) and ("M" not in over or ineq)]
    bad += [{next(a for a in e.args if a in e.bufs): None}, {e.outputs[0]: None}]
    if ineq:
        bad.append(dict(M=1 << 30))                         # M * N overflows int
    return bad


@pytest.mark.parametrize("name", [n + sfx for n in PERCALL for sfx in ("", "_dev")])
def test_per_call_entry_rejects_every_bad_argument_without_a_trace(mpc, traces, name):
    e = percall_entry(mpc, name)
    reject(e, percall_bad(e))
    if not e.dev:
        check_trace(traces[name])


if __name__ == "__main__":
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [root, os.path.join(root, "mpc-ntm-control_b200")]
    import ntm_mpc
    h = ntm_mpc.NtmMpc(0)
    out = {}
    for name in [n for n in FUSED if not n.endswith("_dev")] + list(PERCALL):
        e = fused_entry(h, name) if name in FUSED else percall_entry(h, name)
        try:
            out[name] = trace(e, fused_bad(e.args) if name in FUSED else percall_bad(e))
        except AssertionError as x:                           # reported by the test of that entry
            out[name] = dict(error=str(x)[:1000])
    h.close()
    print(json.dumps(out))
