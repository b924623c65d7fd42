"""CPU: the step_td member of CobelTrace.  The library's struct size and ABI version agree with the ctypes binding,
and every run entry point accepts a trace whose step_td is NULL (argument validation only: nothing is launched)."""
import ctypes as C

import pytest

from cobel_rl_b200 import _lib


@pytest.fixture(scope='module')
def L():
    try:
        return _lib.lib()
    except _lib.CobelError as e:
        pytest.skip(str(e))


def test_trace_layout_and_abi_version(L):
    assert L.cobel_abi_version() == _lib.ABI_VERSION == 6
    assert L.cobel_sizeof(b'CobelTrace') == C.sizeof(_lib.Trace)
    names = [f[0] for f in _lib.Trace._fields_]
    assert names.index('step_td') == names.index('step_next') + 1
    assert _lib.Trace.step_td.offset == _lib.Trace.step_next.offset + 8
    # the positional form of the INTEGRATION.md stub (twelve members) leaves step_td NULL
    tr = _lib.Trace(1, 2, 3, 4, None, 0, None, 0, None, 0, None, None)
    assert tr.step_td is None
    for name, cls in _lib.STRUCTS.items():
        assert L.cobel_sizeof(name.encode()) == C.sizeof(cls), name


@pytest.mark.parametrize('entry,cls', [('cobel_dynaq_run', _lib.DynaQParams), ('cobel_q_run', _lib.QParams),
                                       ('cobel_sr_run', _lib.SRParams), ('cobel_sr_compact_run', _lib.SRCompactParams),
                                       ('cobel_sfma_run', _lib.SFMAParams), ('cobel_pma_run', _lib.PMAParams)])
def test_null_step_td_is_accepted(L, entry, cls):
    """With zero trials and a NULL step_td a run entry point returns COBEL_OK after validating its arguments; an
    invalid field elsewhere is still reported, so the call did reach the validation."""
    fake = 1 << 40          # never dereferenced: a zero-trial call launches nothing
    p = cls()
    p.n_agents = 1
    w = p.world
    w.n_states, w.n_actions, w.n_starts = 4, 4, 1
    w.succ = w.reward = w.terminal = w.starts = fake
    p.stream.draw_count = fake
    p.policy.param = fake
    t = p.trace
    t.trial_steps = t.trial_reward = t.n_steps = t.n_replay = t.flags = fake
    t.step_td = None
    for f, typ in cls._fields_:
        if typ is _lib.c_ptr and getattr(p, f) is None:
            setattr(p, f, fake)
    if hasattr(p, 'mem_policy'):
        p.mem_policy.param = fake
    if hasattr(p, 'n_keys'):
        p.n_keys = 4
    if hasattr(p, 'max_visited'):
        p.max_visited = 4
    p.trials, p.steps = 0, 1
    assert getattr(L, entry)(C.byref(p), None) == 0, entry
    p.n_agents = -1
    assert getattr(L, entry)(C.byref(p), None) < 0, entry
