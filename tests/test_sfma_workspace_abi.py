"""CPU: cobel_sfma_workspace_bytes and the workspace argument of cobel_sfma_run.  SFMA configurations that need the
fused kernel keep its per-agent tables (the SfmaSmem layout of csrc/sfma.cu) in a caller-provided workspace once they
exceed shared memory.  Every run call below is rejected before any kernel launches, so the table pointers may be small
host buffers (validation only checks them for non-NULL)."""
import ctypes

import pytest

EINVAL, EUNSUPPORTED = -1, -2
KMAX_SMEM = 227 * 1024


@pytest.fixture(scope='module')
def L():
    import __graft_entry__ as g
    g.build()
    from cobel_rl_b200 import _lib
    return _lib.lib()


def _params(buf, n_states, n_actions=4, batch=32, **kw):
    """CobelSFMAParams of one agent whose pointers all point at `buf`; the default options take the split path."""
    from cobel_rl_b200 import _lib
    addr = ctypes.addressof(buf)

    def fill(s):
        for name, typ in s._fields_:
            if typ is ctypes.c_void_p:
                setattr(s, name, addr)
            elif issubclass(typ, ctypes.Structure):
                fill(getattr(s, name))
    p = _lib.SFMAParams()
    fill(p)
    p.n_agents, p.trials, p.steps, p.batch, p.nb_replays, p.learn = 1, 1, 1, batch, 1, 1
    p.decay_strength = 1.0
    p.world.n_states, p.world.n_actions, p.world.n_starts = n_states, n_actions, 1
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def sfma_smem_bytes(S, A, T, B, track_t, random_replay):
    """SfmaSmem(S, A, T, B, track_t, random_replay).bytes (csrc/sfma.cu), restated."""
    N = S * A
    t = 3 * N * 8
    r = t + (N * 8 if track_t else 0)
    part = r + N * 8 + S * 8
    rep = part + (T + 32) * 8
    mx = rep + ((B + 1) & ~1) * 4
    mbits = mx + N * 2
    lst = (mbits + S + 3) & ~3
    cdf = (lst + N * 4 + 7) & ~7
    return (cdf + (N * 8 if random_replay else 0) + 15) & ~15


def fused_threads(N):
    return 64 if N <= 128 else 128 if N <= 512 else 256


def _size(L, p):
    return L.cobel_sfma_workspace_bytes(ctypes.byref(p))


def test_size_of_a_50x50_world_with_recency(L):
    buf = ctypes.create_string_buffer(256)
    assert _size(L, _params(buf, 2500, recency=1)) == 484944
    assert sfma_smem_bytes(2500, 4, 256, 32, True, False) == 484944


@pytest.mark.parametrize('options', [
    dict(recency=1), dict(decay_strength=0.95), dict(mod_flags=2), dict(no_replay=1),
    dict(recency=1, learn=0, no_replay=1), dict(decay_strength=0.95, learn=0, no_replay=1),
    dict(recency=1, random_replay=1), dict(mod_flags=2 | 1 | 4 | 8 | 16 | 32)])
@pytest.mark.parametrize('S, A, B', [(2500, 4, 32), (1225, 4, 32), (1444, 4, 32), (600, 8, 16), (4000, 2, 8)])
def test_size_equals_the_fused_layout_beyond_shared_memory(L, options, S, A, B):
    """The fused kernel runs: the size is its SfmaSmem block when that exceeds shared memory, else 0 (on-chip)."""
    buf = ctypes.create_string_buffer(256)
    p = _params(buf, S, A, B, **options)
    track_t = bool(options.get('recency') or options.get('no_replay'))
    want = sfma_smem_bytes(S, A, fused_threads(S * A), B, track_t, bool(options.get('random_replay')))
    assert _size(L, p) == (want if want > KMAX_SMEM else 0)


@pytest.mark.parametrize('S, options, fits', [
    (34 * 34, dict(recency=1), True), (35 * 35, dict(recency=1), False),
    (34 * 34, dict(no_replay=1), True), (35 * 35, dict(no_replay=1), False),
    (34 * 34, dict(learn=0, no_replay=1, decay_strength=0.95), True),
    (35 * 35, dict(learn=0, no_replay=1, decay_strength=0.95), False),
    (37 * 37, dict(decay_strength=0.95), True), (38 * 38, dict(decay_strength=0.95), False),
    (37 * 37, dict(mod_flags=2), True), (38 * 38, dict(mod_flags=2), False)])
def test_boundary_worlds(L, S, options, fits):
    """1191 states with M.T tracked, 1428 without, at 4 actions, 256 threads and a batch of 32."""
    buf = ctypes.create_string_buffer(256)
    size = _size(L, _params(buf, S, **options))
    assert (size == 0) == fits
    if not fits:
        assert size > KMAX_SMEM


@pytest.mark.parametrize('S, options', [
    (2500, dict()), (2500, dict(mod_flags=1 | 4 | 8 | 16 | 32)), (2500, dict(random_replay=1)),
    (32767, dict()), (2500, dict(learn=0, no_replay=1)), (400, dict(recency=1)), (400, dict(decay_strength=0.9))])
def test_size_is_zero_on_the_split_path_and_on_chip(L, S, options):
    """The split path (decay_strength == 1, M.T neither read nor kept, no reward_mod; test() of such a memory takes it
    too) and on-chip fused tables need no workspace."""
    buf = ctypes.create_string_buffer(256)
    assert _size(L, _params(buf, S, **options)) == 0


def _run(L, p):
    before = L.cobel_launch_count()
    rc = L.cobel_sfma_run(ctypes.byref(p), None)
    assert L.cobel_launch_count() == before, 'launched before rejecting the call'
    msg = ctypes.create_string_buffer(512)
    L.cobel_last_error(msg, 512)
    return rc, msg.value.decode()


@pytest.mark.parametrize('options', [dict(recency=1), dict(decay_strength=0.95), dict(mod_flags=2), dict(no_replay=1),
                                     dict(learn=0, no_replay=1, recency=1)])
def test_null_workspace_is_rejected_before_any_launch(L, options):
    buf = ctypes.create_string_buffer(256)
    p = _params(buf, 2500, **options)
    p.workspace = None
    size = _size(L, p)
    assert size > KMAX_SMEM
    rc, msg = _run(L, p)
    assert rc == EINVAL
    assert ('pass a workspace of n_agents x %d bytes' % size) in msg


@pytest.mark.parametrize('options', [dict(), dict(recency=1), dict(decay_strength=0.95)])
def test_more_than_32767_states_is_unsupported(L, options):
    buf = ctypes.create_string_buffer(256)
    p = _params(buf, 32768, **options)
    rc, msg = _run(L, p)
    assert rc == EUNSUPPORTED and msg == 'SFMA kernel supports at most 32767 states'
    assert _size(L, p) == EUNSUPPORTED


def test_query_rejects_bad_arguments(L):
    assert L.cobel_sfma_workspace_bytes(None) == EINVAL
    buf = ctypes.create_string_buffer(256)
    assert _size(L, _params(buf, 0)) == EINVAL
    assert _size(L, _params(buf, 2500, batch=-1)) == EINVAL
