"""ctypes binding of the C ABI declared in include/cobel_b200.h.

There is no CPU fallback: if ``libcobel_b200.so`` has not been built (see
``__graft_entry__.build()``) every compute entry point raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libcobel_b200.so')
ABI_VERSION = 6

c_f64p = C.c_void_p   # device pointers travel as raw addresses
c_ptr = C.c_void_p


class World(C.Structure):
    _fields_ = [('n_states', C.c_int32), ('n_actions', C.c_int32), ('n_starts', C.c_int32),
                ('reserved', C.c_int32), ('succ', c_ptr), ('reward', c_ptr), ('terminal', c_ptr),
                ('starts', c_ptr), ('tp_off', c_ptr), ('tp_next', c_ptr), ('tp_prob', c_ptr)]


class Stream(C.Structure):
    _fields_ = [('seed', C.c_uint64), ('agent_id_base', C.c_int64), ('draw_count', c_ptr),
                ('user_stream', c_ptr), ('user_stream_len', C.c_int64)]


class Policy(C.Structure):
    _fields_ = [('kind', C.c_int32), ('reserved', C.c_int32), ('param', c_ptr)]


class Trace(C.Structure):
    _fields_ = [('trial_steps', c_ptr), ('trial_reward', c_ptr), ('n_steps', c_ptr), ('n_replay', c_ptr),
                ('step_sa', c_ptr), ('step_cap', C.c_int64), ('replay_idx', c_ptr), ('replay_cap', C.c_int64),
                ('replay_len', c_ptr), ('replay_calls_cap', C.c_int64), ('flags', c_ptr), ('step_next', c_ptr),
                ('step_td', c_ptr), ('replay_td', c_ptr)]


class DynaQParams(C.Structure):
    _fields_ = [('n_agents', C.c_int64), ('world', World), ('stream', Stream), ('policy', Policy),
                ('trace', Trace), ('Q', c_ptr), ('Mr', c_ptr), ('Ms', c_ptr), ('Mt', c_ptr),
                ('action_mask', c_ptr), ('mask_agent_stride', C.c_int64), ('lr', c_ptr), ('gamma', c_ptr),
                ('mem_lr', c_ptr), ('trials', C.c_int32), ('steps', C.c_int32), ('batch', C.c_int32),
                ('learn', C.c_int32), ('no_replay', C.c_int32), ('episodic_replay', C.c_int32)]


class QParams(C.Structure):
    _fields_ = [('n_agents', C.c_int64), ('world', World), ('stream', Stream), ('policy', Policy),
                ('trace', Trace), ('Q', c_ptr), ('obs_key', c_ptr), ('n_keys', C.c_int32), ('reserved', C.c_int32),
                ('log', c_ptr), ('log_cap', C.c_int64), ('log_len', c_ptr), ('lr', c_ptr), ('gamma', c_ptr),
                ('trials', C.c_int32), ('steps', C.c_int32), ('batch', C.c_int32), ('learn', C.c_int32)]


class SRParams(C.Structure):
    _fields_ = [('n_agents', C.c_int64), ('world', World), ('stream', Stream), ('policy', Policy),
                ('trace', Trace), ('SR', c_ptr), ('rewards', c_ptr), ('model', c_ptr), ('action_mask', c_ptr),
                ('mask_agent_stride', C.c_int64), ('lr', c_ptr), ('gamma', c_ptr), ('trials', C.c_int32),
                ('steps', C.c_int32), ('learn', C.c_int32), ('reserved', C.c_int32)]


class SRCompactParams(C.Structure):
    _fields_ = [('n_agents', C.c_int64), ('world', World), ('stream', Stream), ('policy', Policy),
                ('trace', Trace), ('SRc', c_ptr), ('rewards', c_ptr), ('model', c_ptr), ('visited', c_ptr),
                ('n_visited', c_ptr), ('action_mask', c_ptr), ('lr', c_ptr), ('gamma', c_ptr),
                ('max_visited', C.c_int32), ('trials', C.c_int32), ('steps', C.c_int32), ('learn', C.c_int32)]


class SFMAParams(C.Structure):
    _fields_ = [('n_agents', C.c_int64), ('world', World), ('stream', Stream), ('policy', Policy),
                ('trace', Trace), ('Q', c_ptr), ('Mr', c_ptr), ('Ms', c_ptr), ('Mt', c_ptr), ('C', c_ptr),
                ('T', c_ptr), ('I', c_ptr), ('D', c_ptr), ('action_mask', c_ptr), ('mask_agent_stride', C.c_int64),
                ('lr', c_ptr), ('gamma', c_ptr), ('mem_lr', c_ptr), ('beta', C.c_double), ('threshold', C.c_double),
                ('decay_inhibition', C.c_double), ('decay_strength', C.c_double), ('decay_recency', C.c_double),
                ('c_step', C.c_double), ('i_step', C.c_double), ('blend', C.c_double), ('interp_fwd', C.c_double),
                ('interp_rev', C.c_double), ('mode', C.c_int32), ('recency', C.c_int32), ('deterministic', C.c_int32),
                ('trials', C.c_int32), ('steps', C.c_int32), ('batch', C.c_int32), ('nb_replays', C.c_int32),
                ('start_replay', C.c_int32), ('random_replay', C.c_int32), ('dynamic', C.c_int32),
                ('no_replay', C.c_int32), ('learn', C.c_int32), ('td_acc', c_ptr), ('trial_mode', c_ptr),
                ('reward_modulation', C.c_double), ('mod_flags', C.c_int32), ('exp_bound', C.c_int32), ('carry', c_ptr),
                ('workspace', c_ptr)]


PMA_MAX_SEQ = 64


class PMAParams(C.Structure):
    _fields_ = [('n_agents', C.c_int64), ('world', World), ('stream', Stream), ('policy', Policy),
                ('mem_policy', Policy), ('trace', Trace), ('Q', c_ptr), ('Mr', c_ptr), ('Ms', c_ptr), ('Mt', c_ptr),
                ('T', c_ptr), ('SR', c_ptr), ('update_mask', c_ptr), ('action_mask', c_ptr),
                ('mask_agent_stride', C.c_int64), ('lr', c_ptr), ('gamma', c_ptr), ('mem_lr', c_ptr), ('lr_q', c_ptr),
                ('gamma_q', c_ptr), ('gamma_sr', c_ptr), ('pow_gamma_sr', c_ptr), ('pow_gamma_q', c_ptr),
                ('pow_stride', C.c_int64), ('min_gap', c_ptr), ('carry', c_ptr), ('need_scratch', c_ptr),
                ('lr_T', C.c_double), ('min_gain', C.c_double),
                ('min_gain_original', C.c_int32), ('trials', C.c_int32), ('steps', C.c_int32), ('batch', C.c_int32),
                ('no_replay', C.c_int32), ('learn', C.c_int32), ('sr_band', C.c_int32), ('options', C.c_int32),
                ('band_scratch', c_ptr), ('n_tab', C.c_int32), ('band_trusted', C.c_int32), ('tab_kind', c_ptr),
                ('tab_param', c_ptr), ('tab_of_agent', c_ptr), ('tab_scratch', c_ptr)]


def pma_tab_doubles(n_actions):
    """COBEL_PMA_TAB_DOUBLES(A) of include/cobel_b200.h."""
    return 3 * (1 << (2 * n_actions)) * n_actions


class Experiences(C.Structure):
    _fields_ = [('batch', C.c_int32), ('reserved', C.c_int32), ('state', c_ptr), ('action', c_ptr), ('reward', c_ptr),
                ('next_state', c_ptr), ('terminal', c_ptr), ('td', c_ptr)]


# COBEL_OP_* (include/cobel_b200.h)
OP_STORE, OP_UPDATE_Q, OP_RETRIEVE_BATCH, OP_REPLAY, OP_RETRIEVE_Q, OP_GATHER, OP_GAIN_BATCH, OP_NEED = range(1, 9)

STRUCTS = {'CobelExperiences': Experiences, 'CobelWorld': World, 'CobelStream': Stream, 'CobelPolicy': Policy, 'CobelTrace': Trace,
           'CobelDynaQParams': DynaQParams, 'CobelQParams': QParams, 'CobelSRParams': SRParams, 'CobelSRCompactParams': SRCompactParams, 'CobelSFMAParams': SFMAParams, 'CobelPMAParams': PMAParams}

_SIGNATURES = {
    'cobel_sizeof': (C.c_size_t, [C.c_char_p]),
    'cobel_abi_version': (C.c_int, []),
    'cobel_last_error': (None, [C.c_char_p, C.c_size_t]),
    'cobel_launch_count': (C.c_int64, []),
    'cobel_draw_uniforms': (C.c_int, [C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, c_ptr, c_ptr]),
    'cobel_stream_next': (C.c_int, [C.POINTER(Stream), C.c_int64, C.c_int64, c_ptr, c_ptr]),
    'cobel_dynaq_run': (C.c_int, [C.POINTER(DynaQParams), c_ptr]),
    'cobel_q_run': (C.c_int, [C.POINTER(QParams), c_ptr]),
    'cobel_sr_run': (C.c_int, [C.POINTER(SRParams), c_ptr]),
    'cobel_sr_compact_run': (C.c_int, [C.POINTER(SRCompactParams), c_ptr]),
    'cobel_sfma_run': (C.c_int, [C.POINTER(SFMAParams), c_ptr]),
    'cobel_sfma_workspace_bytes': (C.c_int64, [C.POINTER(SFMAParams)]),
    'cobel_pma_run': (C.c_int, [C.POINTER(PMAParams), c_ptr]),
    'cobel_env_reset': (C.c_int, [C.POINTER(World), C.POINTER(Stream), C.c_int64, c_ptr, c_ptr]),
    'cobel_env_step': (C.c_int, [C.POINTER(World), C.POINTER(Stream), C.c_int64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    'cobel_policy_probs': (C.c_int, [C.POINTER(Policy), C.c_int64, C.c_int64, C.c_int32, c_ptr, c_ptr, c_ptr, c_ptr]),
    'cobel_policy_select': (C.c_int, [C.POINTER(Policy), C.POINTER(Stream), C.c_int64, C.c_int32, c_ptr, c_ptr, c_ptr, c_ptr]),
    'cobel_dynaq_op': (C.c_int, [C.POINTER(DynaQParams), C.c_int, C.POINTER(Experiences), c_ptr]),
    'cobel_q_op': (C.c_int, [C.POINTER(QParams), C.c_int, C.POINTER(Experiences), c_ptr]),
    'cobel_sr_op': (C.c_int, [C.POINTER(SRParams), C.c_int, C.POINTER(Experiences), c_ptr, c_ptr, c_ptr]),
    'cobel_sr_compact_op': (C.c_int, [C.POINTER(SRCompactParams), C.c_int, C.POINTER(Experiences), c_ptr, C.c_int32,
                                      c_ptr, c_ptr]),
    'cobel_sfma_op': (C.c_int, [C.POINTER(SFMAParams), C.c_int, C.POINTER(Experiences), c_ptr]),
    'cobel_sfma_replay': (C.c_int, [C.POINTER(SFMAParams), c_ptr, C.c_int, c_ptr]),
    'cobel_pma_op': (C.c_int, [C.POINTER(PMAParams), C.c_int, C.POINTER(Experiences), c_ptr, c_ptr, c_ptr]),
    'cobel_pma_replay': (C.c_int, [C.POINTER(PMAParams), c_ptr, C.c_int, c_ptr]),
}

_lib = None


class CobelError(RuntimeError):
    pass


def lib():
    """Load the shared library (once).  Raises if it is missing -- no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CobelError(
                '%s not found: build the CUDA extension first (python -c "import __graft_entry__ as g; '
                'g.build()"); cobel_rl_b200 has no CPU fallback' % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        if L.cobel_abi_version() != ABI_VERSION:
            raise CobelError('ABI version mismatch: library %d, binding %d' % (L.cobel_abi_version(), ABI_VERSION))
        _lib = L
    return _lib


def exported_symbols():
    return list(_SIGNATURES)


def check(rc):
    """Translate a C status into the exception the reference would raise."""
    if rc == 0:
        return
    buf = C.create_string_buffer(512)
    lib().cobel_last_error(buf, 512)
    msg = buf.value.decode()
    if rc == -1:
        raise AssertionError(msg)
    if rc == -2:
        raise NotImplementedError(msg)
    raise CobelError(msg)


def call(name, device, *args):
    """Invoke an entry point with `device` as the current CUDA device (the library launches on the
    current device; the stream passed in `args` must belong to it) and raise on a non-zero status."""
    import torch
    with torch.cuda.device(device):
        check(getattr(lib(), name)(*args))


def ptr(t):
    """Device address of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
