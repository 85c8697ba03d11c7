"""Sharded (multi-device) batches, hy_batch_create_multi(): the lanes of one batch split into contiguous blocks, one
single-device batch + one host thread per block. The property the reference pins for its ensembles
(test/ensemble_propagate.cpp:413-431) is that the partitioning does not change the results: a sharded batch must equal
the unsharded one BIT FOR BIT (state, times, step results, propagate results, Taylor coefficients), including the
reference's global exits of propagate_until() and its last_h semantics, which couple the shards.

The shards may live on the same GPU (device list [0, 0, 0]: what runs on a one-GPU box) or on every GPU of the box
("all")."""
import re

import numpy as np
import pytest

import heyoka_b200 as hb
from common import outer_ss_batch_state, sys_outer_ss, sys_tutorial

pytestmark = pytest.mark.gpu

N_DEVICES = hb.lib.hy_device_count()
SEVERAL_GPUS = pytest.mark.skipif(N_DEVICES < 2, reason="needs two or more GPUs")


def _device_lists():
    # one shard; three shards on one GPU (uneven blocks of lanes); one shard per GPU of the machine
    return [[0], [0, 0, 0], pytest.param(list(range(max(N_DEVICES, 2))), marks=SEVERAL_GPUS)]


def _same(a, b):
    assert np.array_equal(a.state, b.state)
    assert np.array_equal(a.time, b.time) and np.array_equal(a._t_lo, b._t_lo)
    assert np.array_equal(a.last_h, b.last_h)


@pytest.mark.parametrize("devs", _device_lists())
def test_sharded_equals_unsharded_bit_for_bit(devs):
    batch = 37  # not a multiple of the number of shards
    st = outer_ss_batch_state(batch)
    one = hb.taylor_adaptive_batch(sys_outer_ss(), st, batch, high_accuracy=True)
    many = hb.taylor_adaptive_batch(sys_outer_ss(), st, batch, high_accuracy=True, device=devs)
    assert many._b.n_shards == min(len(devs), batch) and one._b.n_shards == 0
    assert many._b.kernel_info()["tape"] == one._b.kernel_info()["tape"] == "nbody"

    # step(), step(max_delta_t), step_backward() with write_tc
    for args in ((), (np.linspace(0.01, 0.5, batch),), (None, True)):
        one.step(*args)
        many.step(*args)
        _same(one, many)
        assert one.step_res == many.step_res
    assert np.array_equal(one.tc, many.tc)
    assert np.array_equal(one.update_d_output(-0.5 * one.last_h, rel_time=True),
                          many.update_d_output(-0.5 * many.last_h, rel_time=True))

    # propagate_until() to per-lane times: early lanes get last_h = 0 relative to the GLOBAL loop length
    tf = np.linspace(3.0, 14.0, batch)[::-1].copy()
    one.propagate_until(tf, write_tc=True)
    many.propagate_until(tf, write_tc=True)
    _same(one, many)
    assert one.propagate_res == many.propagate_res
    assert np.array_equal(one.tc, many.tc)
    assert np.count_nonzero(one.last_h == 0.) >= batch - 4

    # propagate_for() with max_delta_t
    one.propagate_for(2.0, max_delta_t=0.3)
    many.propagate_for(2.0, max_delta_t=0.3)
    _same(one, many)
    assert one.propagate_res == many.propagate_res


@pytest.mark.parametrize("devs", _device_lists())
def test_sharded_global_exits(devs):
    """The iteration limit turns EVERY outcome into step_limit; a non-finite lane in ONE shard stops the lanes of EVERY
    shard at that iteration (src/taylor_adaptive_batch.cpp:1462-1467, :1516-1526)."""
    batch = 9
    st = outer_ss_batch_state(batch)
    tf = np.array([0.5, 100., 100., 2.0, 100., 100., 100., 1.0, 100.])
    one = hb.taylor_adaptive_batch(sys_outer_ss(), st, batch)
    many = hb.taylor_adaptive_batch(sys_outer_ss(), st, batch, device=devs)
    one.propagate_until(tf, max_steps=7)
    many.propagate_until(tf, max_steps=7)
    assert [r[0] for r in many.propagate_res] == [hb.taylor_outcome.step_limit] * batch
    assert one.propagate_res == many.propagate_res
    _same(one, many)

    st2 = st.copy()
    st2[6:9, 7] = st2[0:3, 7]  # lane 7 (last shard) starts from a collision: r^-3 = inf -> NaN
    one = hb.taylor_adaptive_batch(sys_outer_ss(), st2, batch)
    many = hb.taylor_adaptive_batch(sys_outer_ss(), st2, batch, device=devs)
    one.propagate_until(100.)
    many.propagate_until(100.)
    assert many.propagate_res[7][0] == hb.taylor_outcome.err_nf_state
    assert one.propagate_res == many.propagate_res
    ok = [i for i in range(batch) if i != 7]
    assert np.array_equal(one.state[:, ok], many.state[:, ok]) and np.array_equal(one.time[ok], many.time[ok])
    # Every other lane stopped after ONE iteration, far from t = 100.
    assert all(many.propagate_res[i][3] == 1 for i in ok)


def test_sharded_with_parameters_and_time():
    """Runtime parameters and time-dependent right-hand sides are sharded like the state (doc/tut_batch_mode.rst system)."""
    batch = 11
    rng = np.random.default_rng(3)
    st = rng.uniform(-1, 1, (2, batch))
    pars = rng.uniform(0.05, 0.3, (1, batch))
    t0 = rng.uniform(0, 2, batch)
    one = hb.taylor_adaptive_batch(sys_tutorial(), st, batch, pars=pars, time=t0)
    many = hb.taylor_adaptive_batch(sys_tutorial(), st, batch, pars=pars, time=t0, device=[0, 0, 0, 0])
    for ta in (one, many):
        ta.step()
        ta.propagate_for(np.linspace(1.0, 3.0, batch))
    _same(one, many)
    assert one.propagate_res == many.propagate_res
    # (propagate_grid() and continuous output of this sharded batch: tests/test_zz_gpu_late_additions.py)


def test_single_shard_refuses_single_device_calls():
    """A batch made by hy_batch_create_multi() with one device is one shard, and still refuses the entry points that
    only a plain batch has."""
    batch = 8
    b = hb.Batch(hb.Program(sys_outer_ss()), batch, device=[0])
    assert b.n_shards == 1
    for exc, name, call in ((ValueError, "hy_batch_get_ptrs()", lambda: b.ptrs()),
                            (ValueError, "hy_batch_set_stream()", lambda: b.set_stream(0)),
                            (ValueError, "hy_batch_propagate_until_dev()", lambda: b.propagate_until_dev(0)),
                            (NotImplementedError, "propagate_grid()", lambda: b.propagate_grid(np.zeros((1, batch)))),
                            (NotImplementedError, "Continuous output", lambda: b.propagate_until_cout(np.ones(batch)))):
        with pytest.raises(exc, match=re.escape(name + " is not available on a multi-device batch")):
            call()


@pytest.mark.parametrize("devs", [None, [0], [0, 0, 0], pytest.param([0, 1], marks=SEVERAL_GPUS)])
def test_propagate_until_host_one_call(devs):
    """hy_batch_propagate_until_host(): upload + propagate_until + downloads in one call, on one device, on one device in
    three pipelined sub-batches (the same device listed three times) and on two devices: bit-identical to the separate
    calls on a plain batch, global exits included (a non-finite lane in one shard stops the lanes of the others at
    the same iteration; the iteration limit turns every outcome into step_limit), and the reference's errors on the
    times."""
    batch = 50
    st = outer_ss_batch_state(batch)
    P = hb.Program(sys_outer_ss(), high_accuracy=True)
    tf = np.linspace(3., 30., batch)

    def plain(st0, tf_, **kw):
        b = hb.Batch(P, batch)
        z = np.zeros(batch)
        b.upload(st0, None, z, z)
        b.propagate_until(tf_, **kw)
        return b.download() + tuple(b.prop_res())

    def fused(st0, tf_, **kw):
        b = hb.Batch(P, batch) if devs is None else hb.Batch(P, batch, device=devs)
        assert b.n_shards == (0 if devs is None else len(devs))
        s, th, tl = st0.copy(), np.zeros(batch), np.zeros(batch)
        last_h, oc, mn, mx, ns = b.propagate_until_host(s, th, tl, tf_, **kw)
        return (s, th, tl, last_h, oc, mn, mx, ns)

    def same(a, b):
        for x, y in zip(a, b):
            assert np.array_equal(np.asarray(x), np.asarray(y), equal_nan=True)

    same(plain(st, tf), fused(st, tf))
    same(plain(st, tf, max_delta_t=np.full(batch, 0.11)), fused(st, tf, max_delta_t=np.full(batch, 0.11)))
    same(plain(st, tf, max_steps=7), fused(st, tf, max_steps=7))  # iteration limit
    bad = st.copy()
    bad[0:3, 41] = bad[6:9, 41]  # two bodies on top of each other: lane 41 goes non-finite at its first step
    ref, got = plain(bad, tf), fused(bad, tf)
    assert ref[4][41] == hb.taylor_outcome.err_nf_state
    same(ref[1:], got[1:])
    ok = np.arange(batch) != 41
    assert np.array_equal(ref[0][:, ok], got[0][:, ok])
    b = hb.Batch(P, batch) if devs is None else hb.Batch(P, batch, device=devs)
    with pytest.raises(ValueError, match="one of the current times is not finite"):
        b.propagate_until_host(st.copy(), np.full(batch, np.inf), np.zeros(batch), tf)
    with pytest.raises(ValueError, match="non-finite time was passed"):
        b.propagate_until_host(st.copy(), np.zeros(batch), np.zeros(batch), np.full(batch, np.nan))
