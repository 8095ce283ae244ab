"""CPU-only checks of the forward simulator's boundary: rt_forward_simulate refuses bad arguments
before it touches the device, and the Python layer refuses bad shards and templates."""
import ctypes
import os

import numpy as np
import pytest

from raoteh_b200 import _native, lowering, synth


def _args(**kw):
    A = _native.ForwardArgs()
    fake = 0x1000          # never dereferenced: every call below fails its argument checks first
    A.S, A.n_nodes, A.n_ops, A.K, A.mode, A.cap = 4, 3, 3, 1, _native.SIM_HISTORY, 8
    A.n_traj, A.traj_stride, A.obs_stride = 10, 10, 10
    for name in ('program', 'parent', 'length', 'obs_slot', 'Q', 'P', 'obs', 'node_state', 'ev_time',
                 'ev_sb', 'ev_count', 'ev_total', 'status'):
        setattr(A, name, fake)
    for k, v in kw.items():
        setattr(A, k, v)
    return A


@pytest.mark.parametrize('change,code', [
    (dict(S=1), 3), (dict(S=65), 3), (dict(K=0), 1), (dict(K=256), 1), (dict(K=2), 1),
    (dict(mode=2), 1), (dict(program=None), 1), (dict(parent=None), 1), (dict(obs_slot=None), 1),
    (dict(traj_stride=9), 1), (dict(obs_stride=9), 1), (dict(n_ops=0), 1), (dict(n_nodes=1), 1),
    (dict(status=None), 1), (dict(ev_time=None), 1), (dict(Q=None), 1), (dict(cap=0), 1),
    (dict(dwell_sum=0x1000), 1), (dict(time_f64=1, S=7), 3), (dict(time_f64=1, S=9), 3),
    (dict(k=-1), 1), (dict(tmpl=0x1000, tmpl_n_sites=0), 1),
    (dict(mode=_native.SIM_NODES, P=None), 1)])
def test_forward_simulate_argument_errors(change, code):
    if not os.path.exists(_native.LIB_PATH):
        from raoteh_b200 import _build
        _build.build()
    A = _args(**change)
    rc = _native.lib().rt_forward_simulate(ctypes.byref(A), None)
    assert rc == code, (change, rc, _native.lib().rt_last_error_string())
    assert _native.lib().rt_forward_simulate(None, None) == 1


def test_shards_and_templates_are_checked_on_the_host():
    from raoteh_b200 import simulate
    assert simulate._shard(10, 0, None) == (0, 10)
    assert simulate._shard(10, 4, None) == (4, 6)
    for bad in ((10, 4, 7), (10, -1, 3), (10, 0, -1)):
        with pytest.raises(ValueError):
            simulate._shard(*bad)
    parent, length, leaves = synth.random_binary_tree(5, 0.1, np.random.default_rng(0))
    sched = lowering.TreeSchedule(parent, length)
    slot, nodes = simulate._leaf_layout(sched, None, None)
    assert np.array_equal(nodes, sched.leaves) and np.array_equal(slot[nodes], np.arange(len(nodes)))
    with pytest.raises(ValueError):
        simulate._root_tensor([0.5, 0.5], 4, 'cpu')
    with pytest.raises(ValueError):
        simulate._root_tensor([0.0, 0.0], 2, 'cpu')
