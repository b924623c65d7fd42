"""CPU: argument checks of cobel_pma_replay beyond 160 states or 1024 one-step backups, where the stand-alone replay
takes the banded eliminations.  Every call below is rejected before any kernel launches, so the table pointers may be
small host buffers (validation only checks them for non-NULL)."""
import ctypes

import pytest

EINVAL, EUNSUPPORTED = -1, -2


@pytest.fixture(scope='module')
def L():
    import __graft_entry__ as g
    g.build()
    from cobel_rl_b200 import _lib
    return _lib.lib()


def _params(buf, n_states, n_actions, sr_band):
    """CobelPMAParams of one agent whose pointers all point at `buf`."""
    from cobel_rl_b200 import _lib
    addr = ctypes.addressof(buf)

    def fill(s):
        for name, typ in s._fields_:
            if typ is ctypes.c_void_p:
                setattr(s, name, addr)
            elif issubclass(typ, ctypes.Structure):
                fill(getattr(s, name))
    p = _lib.PMAParams()
    fill(p)
    p.n_agents, p.learn, p.batch, p.n_tab = 1, 1, 8, 0
    p.world.n_states, p.world.n_actions, p.world.n_starts = n_states, n_actions, 1
    p.sr_band = sr_band
    return p


def _replay(L, p, buf, update_sr):
    before = L.cobel_launch_count()
    rc = L.cobel_pma_replay(ctypes.byref(p), ctypes.addressof(buf), update_sr, None)
    assert L.cobel_launch_count() == before, 'launched before rejecting the call'
    buf2 = ctypes.create_string_buffer(512)
    L.cobel_last_error(buf2, 512)
    return rc, buf2.value.decode()


@pytest.mark.parametrize('update_sr', [0, 1])
@pytest.mark.parametrize('S, A', [(400, 4), (161, 2), (144, 8)])
def test_big_world_without_band_is_unsupported(L, S, A, update_sr):
    """400 states, 161 states, and 144 states with 1152 backups (BIG by its backups only) have no dense eliminations."""
    buf = ctypes.create_string_buffer(256)
    rc, msg = _replay(L, _params(buf, S, A, -1), buf, update_sr)
    assert rc == EUNSUPPORTED
    assert msg == ('PMA: more than 160 states need the banded update_sr (sr_band >= 0; the dense S x S eliminations are '
                   'register-tiled for S <= 160), got %d states' % S)


def test_refresh_too_large_is_rejected_with_update_sr(L):
    """18 x 25: 450 states at half band 25 -- the final refresh (pma_sr_band_kernel<32>) needs 450 * 66 doubles."""
    buf = ctypes.create_string_buffer(256)
    rc, msg = _replay(L, _params(buf, 450, 4, 25), buf, 1)
    assert rc == EUNSUPPORTED
    assert msg == ('PMA: the final SR refresh of 450 states at half band 25 needs 237600 bytes of shared memory (at most '
                   '232448); beyond 160 states there is no dense update_sr to fall back on')


@pytest.mark.parametrize('S, A', [(513, 2), (529, 4), (400, 8)])
def test_beyond_512_states_or_2048_backups_is_rejected(L, S, A):
    buf = ctypes.create_string_buffer(256)
    rc, msg = _replay(L, _params(buf, S, A, 16), buf, 0)
    assert rc == EUNSUPPORTED
    assert msg == 'PMA kernels support at most 512 states and 2048 one-step backups, got %d states x %d actions' % (S, A)


def test_main_kernel_shared_memory_is_checked(L):
    """512 states at 4 actions: four agents' replay tables exceed the main kernel's shared memory."""
    buf = ctypes.create_string_buffer(256)
    rc, msg = _replay(L, _params(buf, 512, 4, 16), buf, 0)
    assert rc == EUNSUPPORTED
    assert msg == 'PMA: 512 states x 4 actions do not fit in shared memory'


@pytest.mark.parametrize('band, scratch', [(32, True), (16, False)])
def test_band_arguments_are_checked(L, band, scratch):
    buf = ctypes.create_string_buffer(256)
    p = _params(buf, 400, 4, band)
    if not scratch:
        p.band_scratch = None
    rc, msg = _replay(L, p, buf, 0)
    assert rc == EINVAL
    assert msg.startswith('sr_band must be < 0')
