"""GPU tests written at the very end of round 2, after the round's last full run of the GPU suite
(profiles/r2_pytest_gpu_tail.log) and with no GPU time left to run them: the file sorts after the others so that
`pytest -x` reaches them last, and its sections go from new assertions on code that run covered to new code.

1. The GPU against the outputs the reference prints in its tutorials (doc/tut_adaptive.rst, tut_d_output.rst,
   tut_events.rst, tut_ensemble.rst, tut_param.rst, tut_nonauto.rst, tut_adaptive_custom.rst; fixtures
   tests/golden/tut_*.json made by tests/golden/make_golden_from_docs.py). The CPU oracle is held to the same fixtures
   with tighter tolerances in tests/test_oracle_golden.py and tests/test_events_cpu.py.
2. The front ends' host loops on a batch made of shards (hy_batch_create_multi()): event detection and
   propagate_grid() run the reference's lock-step loops on the host (src/taylor_adaptive_batch.cpp:728-1035,
   :1696-2053) over the shards' steps and dense output, and must give what the single-device batch gives.
3. API added last: te_cooldowns / get_te_cooldowns(), get_times() / get_tcs() of the continuous output, the C++
   class's remaining reference members (tests/cpp/test_getters.cpp)."""
import os
import subprocess

import numpy as np
import pytest

import event_cases as ec
import heyoka_b200 as hb
from common import outer_ss_batch_state, sys_outer_ss, sys_tutorial

pytestmark = pytest.mark.gpu


def make(*a, **k):
    return hb.taylor_adaptive_batch(*a, **k)


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / np.abs(b)))


# ---- 1. the reference's tutorial outputs on the GPU (tests/golden/tut_*.json): new assertions on code that the
#         round's full GPU run covered ----
def test_tutorial_adaptive_gpu():
    """doc/tut_adaptive.rst (tutorial/adaptive_basic.cpp), the scalar pendulum as a batch of 3 identical lanes: state after
    one step to the 16 digits the reference prints, step counts 24 / 72 / 97, back at the initial condition after 193
    steps, propagate_grid sample. Same assertions as tests/test_oracle_golden.py::test_tutorial_adaptive."""
    from common import golden, sig_digits_equal, sys_pendulum
    g = golden("tut_adaptive.json")
    TO = hb.taylor_outcome
    OC = {"success": TO.success, "time_limit": TO.time_limit}
    n = 3
    ic = np.array([[g["x0"]] * n, [g["v0"]] * n])
    ta = hb.taylor_adaptive_batch(sys_pendulum(), ic, n)
    ta.step()
    fs = g["first_step"]
    assert [r[0] for r in ta.step_res] == [OC[fs["outcome"]]] * n
    assert sig_digits_equal(ta.last_h, [fs["h"]] * n)
    assert _rel(ta.time, [fs["time"]] * n) < 1e-13
    assert _rel(ta.state, np.array(fs["state"])[:, None] * np.ones(n)) < 1e-13
    assert np.all(ta.state == ta.state[:, :1])
    ta.step_backward()
    assert [r[0] for r in ta.step_res] == [OC[g["step_backward"]["outcome"]]] * n
    assert sig_digits_equal(ta.last_h, [g["step_backward"]["h"]] * n)
    for r in g["clamped_steps"]:
        ta.step([r["limit"]] * n)
        assert [x[0] for x in ta.step_res] == [OC[r["outcome"]]] * n and np.all(ta.last_h == r["h"])
    ta.state[:] = ic
    ta.set_time(0.)
    for r, call in zip(g["propagate"], (lambda: ta.propagate_for(5.), lambda: ta.propagate_until(20.),
                                        lambda: ta.propagate_until(0.))):
        call()
        assert [x[0] for x in ta.propagate_res] == [OC[r["outcome"]]] * n
        assert [x[3] for x in ta.propagate_res] == [r["n_steps"]] * n
        assert sig_digits_equal([x[1] for x in ta.propagate_res], [r["min_h"]] * n)
        assert sig_digits_equal([x[2] for x in ta.propagate_res], [r["max_h"]] * n)
        assert np.all(ta.time == r["time"])
    assert _rel(ta.state, np.array(g["state_back_at_0"])[:, None] * np.ones(n)) < 1e-12
    ta.state[:] = ic
    ta.set_time(0.)
    out = ta.propagate_grid(np.array(g["grid"]["times"])[:, None] * np.ones(n))
    k = g["grid"]["index"]
    assert sig_digits_equal(out[k, 0], [g["grid"]["x"]] * n) and sig_digits_equal(out[k, 1], [g["grid"]["v"]] * n)


def test_tutorial_dense_and_continuous_output_gpu():
    """doc/tut_d_output.rst (tutorial/d_output.cpp): dense output after one step, continuous output of
    propagate_until(10): 48 recorded steps, the six printed samples."""
    from common import golden, sig_digits_equal, sys_pendulum
    g = golden("tut_d_output.json")
    ic = np.array([[g["x0"]] * 2, [g["v0"]] * 2])
    ta = hb.taylor_adaptive_batch(sys_pendulum(), ic, 2)
    ta.step(write_tc=True)
    assert np.all(ta.tc[:, 0, :] == ic)
    d = ta.update_d_output(0.1).copy()
    assert sig_digits_equal(d[:, 0], g["d_output_at_0.1"]) and sig_digits_equal(d[:, 1], g["d_output_at_0.1"])
    assert _rel(ta.update_d_output(ta.time), ta.state) < 1e-14
    ta.state[:] = ic
    ta.set_time(0.)
    co = ta.propagate_until(g["c_output"]["t_final"], c_output=True)
    assert co.get_n_steps() == g["c_output"]["n_steps"] == 48
    lb, ub = co.get_bounds()
    assert np.all(lb == 0) and np.all(ub == 10)
    for tm, x, v in g["c_output"]["samples"]:
        s = co(tm)
        assert sig_digits_equal(s[0], [x] * 2) and sig_digits_equal(s[1], [v] * 2), tm


def test_tutorial_events_golden_gpu():
    """doc/tut_events.rst (tutorial/event_basic.cpp): the event times and the grid output the reference prints with 16
    digits, through the device's event detection (tests/event_cases.py::case_tutorial_events, also run on the oracle)."""
    from common import golden
    ec.case_tutorial_events(make, golden("tut_events.json"), loose=50.)


def test_more_tutorials_gpu():
    """The remaining printed outputs of the reference's tutorials on the GPU (same fixtures as tests/test_oracle_golden.py; the tolerances are wider
    than the oracle's because the device's sin / cos differ from the host library's by an ulp or two per call): doc/tut_ensemble.rst (members as lanes, also sharded), doc/tut_param.rst,
    doc/tut_nonauto.rst, doc/tut_adaptive_custom.rst."""
    from common import golden, sig_digits_equal, sys_pendulum
    TO = hb.taylor_outcome
    # Ensemble: member 9 after propagate_until(20): 17 printed digits, 124 steps.
    g = golden("tut_ensemble.json")
    ics = np.array(g["ics"]).T.copy()
    for kw in ({}, {"device": [0, 0, 0]}):
        ta = hb.taylor_adaptive_batch(sys_pendulum(), ics, g["n_iter"], **kw)
        ta.propagate_until(g["t_final"])
        m = g["member"]
        oc, mn, mx, ns = ta.propagate_res[m]
        assert np.all(ta.time == g["time"]) and oc == TO.time_limit and ns == g["n_steps"]
        assert sig_digits_equal(mn, g["min_h"]) and sig_digits_equal(mx, g["max_h"])
        assert _rel(ta.state[:, m], g["state"]) < 1e-12
    # Runtime parameters: back at (0.05, 0) after one period, for two values of the gravitational acceleration.
    g = golden("tut_param.json")
    x, v = hb.make_vars("x", "v")
    runs = g["runs"]
    ta = hb.taylor_adaptive_batch([(x, v), (v, -hb.par[0] / hb.par[1] * hb.sin(x))], [[g["x0"]] * 2, [g["v0"]] * 2], 2,
                                  pars=np.array([r["pars"] for r in runs]).T.copy())
    ta.propagate_until([r["t_final"] for r in runs])
    for i, r in enumerate(runs):
        assert abs(ta.state[0, i] - r["state"][0]) < 1e-14 and abs(ta.state[1, i] - r["state"][1]) < 1e-13
    # Time-dependent right-hand side: 25 printed values of x.
    g = golden("tut_nonauto.json")
    ta = hb.taylor_adaptive_batch([(x, v), (v, hb.cos(hb.time) - .1 * v - hb.sin(x))], [[g["x0"]], [g["v0"]]], 1)
    for k, xr in enumerate(g["x"]):
        ta.propagate_for(g["delta_t"])
        assert sig_digits_equal(ta.state[0, 0], xr), k
    assert ta.time[0] == 50.
    # tol = 1e-9: order 12, the printed state after 0 -> 10 -> 0.
    g = golden("tut_adaptive_custom.json")
    ta = hb.taylor_adaptive_batch(sys_pendulum(), [[g["x0"]], [g["v0"]]], 1, tol=g["tol"])
    assert ta.get_order() == 12
    for tf in g["times"]:
        ta.propagate_until(tf)
    assert np.max(np.abs(ta.state[:, 0] - np.array(g["state_back_at_0"]))) < 1e-13


@pytest.mark.parametrize("case", [ec.case_step_count_te_stop_bug, ec.case_callback_ste, ec.case_propagate_grid_ste,
                                  ec.case_ev_inf_state, ec.case_event_cb_time, ec.case_ev_exception_callback,
                                  ec.case_events_error, ec.case_get_set_dtime, ec.case_reset_cooldowns,
                                  ec.case_param_deduction_from_events], ids=lambda f: f.__name__)
def test_reference_regression_cases_gpu(case):
    """Regression cases of test/taylor_adaptive_batch.cpp (:1456-1471, :1560-1640, :1819-1862, :1944-1980, :2011-2046) for the
    host loops of integrators with events, on the device (tests/test_events_cpu.py runs them on the oracle)."""
    case(make)


def test_step_callback_must_not_alter_the_time_gpu():
    """:2141-2176 "bug prop_cb time": a step callback of propagate_until() that alters the time coordinate - of every
    batch element or of one - is an error."""
    x, v = hb.make_vars("x", "v")
    msg = ("The invocation of the callback passed to propagate_until\\(\\) resulted in the alteration of the time "
           "coordinate of the integrator - this is not supported")

    def all_lanes(t):
        t.set_time(100.)
        return True

    def one_lane(t):
        t.set_time([t.time[0], 100.])
        return True

    for cb in (all_lanes, one_lane):
        ta = hb.taylor_adaptive_batch([(x, v), (v, -x)], [0., 0.1, 1., 1.1], 2)
        with pytest.raises(RuntimeError, match=msg):
            ta.propagate_until(10., callback=cb)


# ---- 2. front-end host loops on sharded batches (written after the round's last full GPU run) ----
def test_sharded_event_batch_equals_single_device():
    """Events on a batch made of shards (hy_batch_create_multi(): here three shards on one GPU, uneven blocks of lanes):
    every shard detects the events of its own lanes, the records come back with the lanes of the whole batch in the same
    order. Bit for bit what the single-device batch produces over 40 lock-step steps with two terminal and two
    non-terminal events (event lists with times, outcomes, step sizes, states, times, Taylor coefficients of the event
    equations, cooldown state), propagate_until() and propagate_grid() through the front end's host loops, and the
    reference-side fixtures of test/batch_event_detection.cpp on the sharded batch."""
    x, v, sys = ec.pendulum_sys()
    batch = 37
    rng = np.random.default_rng(17)
    st = np.stack([rng.uniform(-0.5, 0.5, batch), rng.uniform(-1.0, 1.0, batch)])

    def build(**kw):
        return make(sys, st, batch, t_events=[hb.t_event_batch(v, callback=lambda ta, s, i: True),
                                              hb.t_event_batch(x - 0.1, callback=lambda ta, s, i: True, cooldown=0.05,
                                                               direction=hb.event_direction.positive)],
                    nt_events=[hb.nt_event_batch(v * v - 1e-2, lambda ta, t, s, i: None),
                               hb.nt_event_batch(x * v + 0.05 * hb.cos(hb.time), lambda ta, t, s, i: None,
                                                 direction=hb.event_direction.negative)], **kw)

    one, many = build(), build(device=[0, 0, 0])
    assert many._b.n_shards == 3 and one._b.n_shards == 0
    n_events = 0
    for it in range(40):
        one.step()
        many.step()
        assert one._b.events() == many._b.events(), it
        n_events += len(one._b.events())
        assert one.step_res == many.step_res
        assert np.array_equal(one.state, many.state) and np.array_equal(one.time, many.time)
        assert np.array_equal(one._b.tc_events(4), many._b.tc_events(4))
        for a, b in zip(one._b.cooldowns(2), many._b.cooldowns(2)):
            assert np.array_equal(a, b)
    assert n_events > batch
    one.propagate_until(one.time + 3.0)
    many.propagate_until(many.time + 3.0)
    assert one.propagate_res == many.propagate_res and np.array_equal(one.state, many.state)
    many.reset_cooldowns(5)
    many.reset_cooldowns()
    assert not np.any(many._b.cooldowns(2)[0])
    # The reference's fixtures on the sharded batch.
    sharded = lambda *a, **k: make(*a, device=[0, 0, 0], **k)  # noqa: E731
    times = ec.case_linear_box(sharded)
    assert np.allclose(sorted(times), [1 / 8., 1 / 4., 1 / 2., 1.], rtol=1e-15)
    ec.case_multizero(sharded)
    ec.case_nte_basic(sharded)
    ec.case_te_basic(sharded)
    ec.case_te_propagate_grid(sharded)


def test_propagate_grid_on_a_sharded_batch():
    """propagate_grid() of a batch made of shards (the front end's host loop over the shards' steps and dense output)
    against the device-resident grid loop of the single-device batch: same step counts, same samples (to 1e-13: one
    evaluates the dense output at absolute times, the other at offsets from the start of the step)."""
    batch, n_pts = 21, 40
    st = outer_ss_batch_state(batch)
    grid = np.linspace(0., 15., n_pts)[:, None] * np.linspace(1., 1.3, batch)[None, :]
    one = hb.taylor_adaptive_batch(sys_outer_ss(), st, batch, high_accuracy=True)
    many = hb.taylor_adaptive_batch(sys_outer_ss(), st, batch, high_accuracy=True, device=[0, 0, 0])
    a, b = one.propagate_grid(grid), many.propagate_grid(grid)
    assert a.shape == b.shape == (n_pts, 36, batch)
    # (Relative to the amplitude of each variable over the grid: a coordinate that crosses zero at a grid point would
    # otherwise turn one unit in the last place of the amplitude into a large relative error.)
    scale = np.max(np.abs(a), axis=0, keepdims=True)
    assert np.max(np.abs(a - b) / scale) < 1e-13
    assert [r[0] for r in one.propagate_res] == [r[0] for r in many.propagate_res]
    assert [r[3] for r in one.propagate_res] == [r[3] for r in many.propagate_res]
    assert np.array_equal(one.time, many.time) and np.max(np.abs(one.state - many.state)) == 0.


def test_sharded_grid_and_continuous_output_with_parameters():
    """The tutorial system (runtime parameter, per-lane start times) on four shards: propagate_grid() runs the front
    end's host loop and agrees with the single-device batch; continuous output is single-device only and says so."""
    batch = 11
    rng = np.random.default_rng(3)
    st = rng.uniform(-1, 1, (2, batch))
    pars = rng.uniform(0.05, 0.3, (1, batch))
    t0 = rng.uniform(0, 2, batch)
    one = hb.taylor_adaptive_batch(sys_tutorial(), st, batch, pars=pars, time=t0)
    many = hb.taylor_adaptive_batch(sys_tutorial(), st, batch, pars=pars, time=t0, device=[0, 0, 0, 0])
    for ta in (one, many):
        ta.step()
    g = np.array([many.time, many.time + 0.5, many.time + 1.0])
    assert np.max(np.abs(many.propagate_grid(g) - one.propagate_grid(g))) < 1e-13
    with pytest.raises(NotImplementedError, match="multi-device"):
        many.propagate_until(many.time + 1.0, c_output=True)


# ---- 3. API added after the round's last full GPU run ----
def test_te_cooldowns_property():
    """te_cooldowns of the Python front end (the reference's get_te_cooldowns()) on the device, single and sharded."""
    ec.case_te_cooldowns_property(make)
    ec.case_te_cooldowns_property(lambda *a, **k: make(*a, device=[0, 0], **k))


def test_continuous_output_times_and_tcs():
    """get_times() / get_tcs() of the continuous output (src/continuous_output.cpp:1157-1169; hy_cout_download()):
    layouts, consistency with the object's own evaluation, with the integrator's final Taylor coefficients, and against
    the oracle's recording of the same propagation.

    get_times() returns the high parts of the double-length times the output searches and evaluates with. Where the
    start of an iteration is a plain double (low part 0), the output at get_times()[k] IS the order-0 coefficients of
    iteration k, bit for bit. Elsewhere it is evaluated at h = -lo (or, for lo > 0, at the end of iteration k - 1), as
    in the reference, and agrees with them to a few units in the last place."""
    import oracle
    from test_oracle_golden import cout_fixture, sys_oscillator
    ic, final_tm, _ = cout_fixture()
    P = hb.Program(sys_oscillator())
    ta = hb.taylor_adaptive_batch(sys_oscillator(), ic, 4)
    t0 = np.array(ta.time)
    co = ta.propagate_until(final_tm, c_output=True)
    n = co.get_n_steps()
    tms, tcs = co.get_times(), co.get_tcs()
    assert tms.shape == (n + 2, 4) and tcs.shape == (n, P.n_eq, P.order + 1, 4)
    assert np.array_equal(tms[0], t0) and np.array_equal(tms[n], final_tm) and np.all(tms[n + 1] == np.inf)
    lb, ub = co.get_bounds()
    assert np.array_equal(lb, tms[0]) and np.array_equal(ub, tms[n])
    assert np.all(np.diff(tms[:n + 1], axis=0) >= 0)
    tms_lo = np.empty_like(tms)
    hb.check(hb.lib.hy_cout_download(co._h, None, hb._dptr(tms_lo), None))
    rounding = 4 * np.finfo(np.float64).eps * np.max(np.abs(tcs[:, :, 0, :]), axis=0)
    n_exact = 0
    for k in range(n):
        out, c0, exact = co(tms[k]), tcs[k][:, 0, :], tms_lo[k] == 0
        assert np.array_equal(out[:, exact], c0[:, exact]), k
        # (An offset of lo in time: first order in lo, plus rounding.)
        assert np.all(np.abs(out - c0) <= 2 * np.abs(tcs[k][:, 1, :] * tms_lo[k]) + rounding), k
        n_exact += int(np.sum(exact))
    assert n_exact >= 4  # (every lane starts at a plain double)
    assert np.array_equal(tcs[n - 1], ta.tc)
    o = oracle.OracleIntegrator(P, ic, 4, mode=oracle.FMA)
    oco = o.propagate_until_cout(final_tm)
    assert oco.get_n_steps() == n
    assert np.max(np.abs(tms[:n + 1] - oco.t_hi[:n + 1])) < 1e-12 and np.array_equal(tms[n + 1], oco.t_hi[n + 1])
    scale = np.max(np.abs(oco.tcs), axis=(0, 1, 3), keepdims=True)
    assert np.max(np.abs(tcs - oco.tcs) / scale) < 1e-11


def test_cpp_late_getters():
    """is_variational(), get_n_orig_sv(), get_dtime_data(), get_state_range() / get_pars_range(), get_te_cooldowns() of
    the drop-in C++ class (include/heyoka/taylor.hpp:961-996 in the reference)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src, lib = os.path.join(root, "tests", "cpp", "test_getters.cpp"), os.path.join(root, "heyoka_b200", "lib")
    exe = os.path.join(root, "build", "test_getters")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    subprocess.run(["g++", "-std=c++17", "-O1", "-I" + os.path.join(root, "include"), src, "-o", exe, "-L" + lib,
                    "-lheyoka_b200", "-Wl,-rpath," + lib], check=True)
    res = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "ALL PASSED (getters)" in res.stdout, res.stdout[-3000:] + res.stderr[-2000:]
