"""CPU: the replay_td member of CobelTrace.  It takes the place of the former padding pointer, so the struct size, every
offset and the ABI version stay as they were; every run entry point accepts a NULL replay_td and rejects a replay_td
without replay_idx before any launch (argument validation only: zero-trial calls launch nothing)."""
import ctypes as C

import pytest

from cobel_rl_b200 import _lib

EINVAL = -1
ENTRIES = [('cobel_dynaq_run', _lib.DynaQParams), ('cobel_q_run', _lib.QParams), ('cobel_sr_run', _lib.SRParams),
           ('cobel_sr_compact_run', _lib.SRCompactParams), ('cobel_sfma_run', _lib.SFMAParams),
           ('cobel_pma_run', _lib.PMAParams)]


@pytest.fixture(scope='module')
def L():
    try:
        return _lib.lib()
    except _lib.CobelError as e:
        pytest.skip(str(e))


def test_trace_layout_and_abi_version(L):
    assert L.cobel_abi_version() == _lib.ABI_VERSION == 6
    names = [f[0] for f in _lib.Trace._fields_]
    assert names[-1] == 'replay_td' and 'reserved' not in names
    assert _lib.Trace.replay_td.offset == _lib.Trace.step_td.offset + 8 == 104
    assert C.sizeof(_lib.Trace) == L.cobel_sizeof(b'CobelTrace') == 112
    for name, cls in _lib.STRUCTS.items():
        assert L.cobel_sizeof(name.encode()) == C.sizeof(cls), name
    # the thirteen-member positional form (before replay_td had a name) leaves it NULL
    tr = _lib.Trace(1, 2, 3, 4, None, 0, None, 0, None, 0, None, None, None)
    assert tr.replay_td is None


def _zero_trial_params(cls):
    """A parameter struct that passes every argument check of its run entry point with zero trials; the trace's
    optional buffers, replay_idx and replay_td included, are NULL."""
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
    return p, fake


@pytest.mark.parametrize('entry,cls', ENTRIES)
def test_null_replay_td_is_accepted(L, entry, cls):
    p, fake = _zero_trial_params(cls)
    assert p.trace.replay_td is None
    assert getattr(L, entry)(C.byref(p), None) == 0, entry
    p.trace.replay_idx = fake
    assert getattr(L, entry)(C.byref(p), None) == 0, entry
    p.trace.replay_td = fake
    assert getattr(L, entry)(C.byref(p), None) == 0, entry


@pytest.mark.parametrize('entry,cls', ENTRIES)
def test_replay_td_without_replay_idx_is_rejected(L, entry, cls):
    p, fake = _zero_trial_params(cls)
    p.trace.replay_td = fake
    before = L.cobel_launch_count()
    assert getattr(L, entry)(C.byref(p), None) == EINVAL, entry
    buf = C.create_string_buffer(256)
    L.cobel_last_error(buf, 256)
    assert buf.value.decode() == 'trace.replay_td needs trace.replay_idx'
    p.trials = 1                            # rejected before the launch of a non-empty call too
    assert getattr(L, entry)(C.byref(p), None) == EINVAL, entry
    assert L.cobel_launch_count() == before
    # the other argument checks come first: their messages are unchanged
    p.trials, p.n_agents = 0, -1
    assert getattr(L, entry)(C.byref(p), None) == EINVAL
    L.cobel_last_error(buf, 256)
    assert buf.value.decode() == 'n_agents must be positive'
