"""CPU: the C-ABI library builds, loads and exports every symbol include/cobel_b200.h declares
(no compute call is made -- there is no GPU here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def built():
    import __graft_entry__ as g
    g.build()
    return ctypes.CDLL(g.LIB)


def declared_functions():
    text = open(os.path.join(ROOT, 'include', 'cobel_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(cobel_[a-z0-9_]+)\s*\(', text)))


def test_header_symbols_exported(built):
    names = declared_functions()
    assert 'cobel_dynaq_run' in names
    for n in names:
        assert hasattr(built, n), 'missing export %s' % n


def test_binding_covers_header(built):
    from cobel_rl_b200 import _lib
    assert sorted(_lib.exported_symbols()) == declared_functions()
    assert built.cobel_abi_version() == _lib.ABI_VERSION


def test_struct_sizes_match(built):
    """ctypes mirrors must have the C layout: compare against sizes the library reports."""
    from cobel_rl_b200 import _lib
    built.cobel_sizeof.restype = ctypes.c_size_t
    built.cobel_sizeof.argtypes = [ctypes.c_char_p]
    for name, cls in _lib.STRUCTS.items():
        assert built.cobel_sizeof(name.encode()) == ctypes.sizeof(cls), name


def test_no_fallback_without_library(monkeypatch):
    from cobel_rl_b200 import _lib
    monkeypatch.setattr(_lib, '_lib', None)
    monkeypatch.setattr(_lib, 'LIB_PATH', '/nonexistent/libcobel_b200.so')
    with pytest.raises(_lib.CobelError):
        _lib.lib()


def test_integration_md_stub_matches_library(built, monkeypatch):
    """The ctypes stub shown in INTEGRATION.md must mirror the header: execute its struct definitions
    against the built library (its own cobel_sizeof assertion runs)."""
    import __graft_entry__ as g
    text = open(os.path.join(ROOT, 'INTEGRATION.md')).read()
    block = text.split('```python')[2].split('```')[0]
    defs = block.split('def dynaq_train_b200')[0]
    monkeypatch.setenv('COBEL_B200_LIB', g.LIB)
    ns = {}
    exec(compile(defs, 'INTEGRATION.md', 'exec'), ns)
    assert ctypes.sizeof(ns['DynaQParams']) == built.cobel_sizeof(b'CobelDynaQParams')


# ---- argument checks of the entry points: every call below is rejected before any kernel launches, so the table
# pointers may be small host buffers (validation only checks them for non-NULL) ---------------------------------------
EINVAL, EUNSUPPORTED = -1, -2


def _params(cls, buf, n_actions):
    """A parameter struct whose pointers (nested structs included) all point at `buf`, with valid sizes."""
    def fill(s):
        for name, typ in s._fields_:
            if typ is ctypes.c_void_p:
                setattr(s, name, ctypes.addressof(buf))
            elif issubclass(typ, ctypes.Structure):
                fill(getattr(s, name))
    p = cls()
    fill(p)
    p.n_agents = 1
    p.world.n_states, p.world.n_actions, p.world.n_starts = 4, n_actions, 1
    for name, value in (('trials', 1), ('steps', 1), ('learn', 1), ('n_keys', 4), ('log_cap', 1), ('max_visited', 4),
                        ('sr_band', -1)):
        if hasattr(p, name):
            setattr(p, name, value)
    return p


def _last_error(L):
    buf = ctypes.create_string_buffer(512)
    L.cobel_last_error(buf, 512)
    return buf.value.decode()


@pytest.mark.parametrize('entry, struct, replay', [
    ('cobel_dynaq_run', 'DynaQParams', False), ('cobel_q_run', 'QParams', False), ('cobel_sr_run', 'SRParams', False),
    ('cobel_sr_compact_run', 'SRCompactParams', False), ('cobel_sfma_run', 'SFMAParams', False),
    ('cobel_pma_run', 'PMAParams', False), ('cobel_sfma_replay', 'SFMAParams', True),
    ('cobel_pma_replay', 'PMAParams', True)])
def test_unsupported_action_count(built, entry, struct, replay):
    from cobel_rl_b200 import _lib
    L = _lib.lib()
    buf = ctypes.create_string_buffer(256)
    p = _params(getattr(_lib, struct), buf, 5)
    args = (ctypes.addressof(buf), 1) if replay else ()
    assert getattr(L, entry)(ctypes.byref(p), *args, None) == EUNSUPPORTED
    assert _last_error(L) == 'unsupported number of actions 5 (built for 2,3,4,6,8)'


def test_sfma_run_requires_carry(built):
    from cobel_rl_b200 import _lib
    L = _lib.lib()
    buf = ctypes.create_string_buffer(256)
    p = _params(_lib.SFMAParams, buf, 4)
    p.trials, p.carry = 0, None
    assert L.cobel_sfma_run(ctypes.byref(p), None) == EINVAL


def test_pma_band_refresh_too_large_is_rejected_before_any_launch(built):
    """Half bands 25..31 beyond 440 states: the final SR refresh (pma_sr_band_kernel<32>, S * 66 doubles of shared
    memory) does not fit, and more than 160 states have no dense update_sr.  cobel_pma_run must say so before its
    first launch, so that a failed call leaves Q, T and the random stream as they were."""
    from cobel_rl_b200 import _lib
    L = _lib.lib()
    buf = ctypes.create_string_buffer(256)
    p = _params(_lib.PMAParams, buf, 4)
    p.world.n_states, p.sr_band = 450, 25
    before = L.cobel_launch_count()
    assert L.cobel_pma_run(ctypes.byref(p), None) == EUNSUPPORTED
    assert _last_error(L) == ('PMA: the final SR refresh of 450 states at half band 25 needs 237600 bytes of shared '
                              'memory (at most 232448); beyond 160 states there is no dense update_sr to fall back on')
    assert L.cobel_launch_count() == before
