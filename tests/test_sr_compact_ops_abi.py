"""CPU: argument checks of cobel_sr_compact_op (stand-alone SR.update / SR.retrieve_q on the compact tables).
Every call below is rejected before any kernel launches, so the table pointers may be small host buffers
(validation only checks them for non-NULL)."""
import ctypes

import pytest

EINVAL, EUNSUPPORTED = -1, -2
STORE, RETRIEVE_Q = 1, 5


@pytest.fixture(scope='module')
def L():
    import __graft_entry__ as g
    g.build()
    from cobel_rl_b200 import _lib
    return _lib.lib()


def _params(buf, n_actions=4, n_states=4, max_visited=4):
    """CobelSRCompactParams whose pointers all point at `buf`."""
    from cobel_rl_b200 import _lib
    addr = ctypes.addressof(buf)
    p = _lib.SRCompactParams()
    for name in ('SRc', 'rewards', 'model', 'visited', 'n_visited', 'lr', 'gamma'):
        setattr(p, name, addr)
    p.stream.draw_count = addr
    p.trace.flags = addr
    p.n_agents, p.max_visited = 1, max_visited
    p.world.n_states, p.world.n_actions = n_states, n_actions
    return p


def _experiences(buf):
    from cobel_rl_b200 import _lib
    a = ctypes.addressof(buf)
    return _lib.Experiences(1, 0, a, a, a, a, a, None)


def _call(L, p, op, buf):
    a = ctypes.addressof(buf)
    if op == STORE:
        return L.cobel_sr_compact_op(ctypes.byref(p), op, ctypes.byref(_experiences(buf)), None, 0, None, None)
    return L.cobel_sr_compact_op(ctypes.byref(p), op, None, a, 1, a, None)


def _last_error(L):
    buf = ctypes.create_string_buffer(512)
    L.cobel_last_error(buf, 512)
    return buf.value.decode()


@pytest.mark.parametrize('op', [STORE, RETRIEVE_Q])
def test_unsupported_action_count(L, op):
    buf = ctypes.create_string_buffer(256)
    assert _call(L, _params(buf, n_actions=5), op, buf) == EUNSUPPORTED
    assert _last_error(L) == 'unsupported number of actions 5 (built for 2,3,4,6,8)'


@pytest.mark.parametrize('missing', ['SRc', 'rewards', 'model', 'visited', 'n_visited', 'lr', 'gamma'])
def test_missing_tables(L, missing):
    buf = ctypes.create_string_buffer(256)
    p = _params(buf)
    setattr(p, missing, None)
    for op in (STORE, RETRIEVE_Q):
        assert _call(L, p, op, buf) == EINVAL
        assert _last_error(L) == 'agent tables missing'


def test_bad_max_visited_op_and_arguments(L):
    buf = ctypes.create_string_buffer(256)
    for v in (1, 65536):
        assert _call(L, _params(buf, max_visited=v), RETRIEVE_Q, buf) == EINVAL
        assert _last_error(L) == 'max_visited must be in 2..65535'
    p = _params(buf)
    a = ctypes.addressof(buf)
    for op in (2, 3, 4, 8):                                          # ops of the other agents
        assert L.cobel_sr_compact_op(ctypes.byref(p), op, ctypes.byref(_experiences(buf)), a, 1, a, None) == EINVAL
    assert L.cobel_sr_compact_op(ctypes.byref(p), RETRIEVE_Q, None, a, 0, a, None) == EINVAL   # n_query = 0
    assert L.cobel_sr_compact_op(ctypes.byref(p), RETRIEVE_Q, None, None, 1, a, None) == EINVAL
    assert L.cobel_sr_compact_op(ctypes.byref(p), STORE, None, None, 0, None, None) == EINVAL


def test_slot_map_too_large_is_rejected_before_any_launch(L):
    """120 000 states: the uint16 slot map alone (240 000 bytes) exceeds the 227 KB of shared memory of one block.
    RETRIEVE_Q also needs the list of reward-carrying columns, min(max_visited, S) uint16 entries, which sets a
    lower limit (58 104 states when max_visited >= S).  Both are refused by name, before anything launches."""
    buf = ctypes.create_string_buffer(256)
    before = L.cobel_launch_count()
    assert _call(L, _params(buf, n_states=120000, max_visited=4), STORE, buf) == EUNSUPPORTED
    assert _last_error(L) == ('cobel_sr_compact_op(STORE): the slot map of 120000 states needs 240032 bytes of shared '
                              'memory (at most 232448)')
    assert _call(L, _params(buf, n_states=120000, max_visited=4), RETRIEVE_Q, buf) == EUNSUPPORTED
    assert _last_error(L) == ('cobel_sr_compact_op(RETRIEVE_Q): the slot map of 120000 states and the list of up to 4 '
                              'reward-carrying states need 240040 bytes of shared memory (at most 232448)')
    assert _call(L, _params(buf, n_states=60000, max_visited=60000), RETRIEVE_Q, buf) == EUNSUPPORTED
    assert _last_error(L) == ('cobel_sr_compact_op(RETRIEVE_Q): the slot map of 60000 states and the list of up to '
                              '60000 reward-carrying states need 240032 bytes of shared memory (at most 232448)')
    assert L.cobel_launch_count() == before
