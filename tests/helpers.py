"""Shared helpers of the parity tests: run one case of oracle/cases.py through the
oracle (CPU) or through the CUDA path, and compare records field by field."""
import os

import numpy as np

from oracle import cases, tabular as tb
from oracle.philox import LazyStream

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')

TRAJ = ['states', 'actions', 'next_states', 'rewards', 'trial_steps', 'trial_reward']
KEYS = {
    'dynaq': TRAJ + ['replay', 'replay_len', 'Q', 'Mr', 'Ms', 'Mt', 'draws'],
    'q_grid': TRAJ + ['replay', 'replay_len', 'Q', 'draws'],
    'q_topo': TRAJ + ['replay', 'replay_len', 'Q', 'draws'],
    'sr': TRAJ + ['SR', 'rew', 'model', 'draws'],
    'sfma': TRAJ + ['replay', 'replay_len', 'Q', 'Mr', 'Ms', 'Mt', 'C', 'T', 'I', 'draws'],
    'pma': TRAJ + ['replay', 'replay_len', 'Q', 'Mr', 'Ms', 'Mt', 'T', 'SR', 'update_mask', 'draws'],
}


def load_golden(name):
    with np.load(os.path.join(GOLDEN, name + '.npz')) as z:
        return {k: z[k] for k in z.files}


# --------------------------------------------------------------------------- #
# recorded values of the parity checks against the reference
# --------------------------------------------------------------------------- #
# The reference sources are not part of this repository.  Its tests/test_oracle_vs_reference.py and the reference
# comparisons of the *_cpu tests therefore check against values stored under tests/golden/: whole records as arrays
# (recorded_records.npz) and everything else in a canonical JSON form (recorded_values.json).
#
# Provenance: these values were NOT produced by the reference.  They were recorded (COBEL_RECORD_REFERENCE=ours) from
# this repository's own oracle and product code at commit 0d657d9, whose oracle/ and product code are identical to
# commit b46dadc, where the same comparisons ran live against the unmodified reference and passed.  They are believed
# equal to what the reference returns but were never checked against it; until they are re-recorded from the reference
# (COBEL_RECORD_REFERENCE=reference, with its sources importable through oracle/ref_loader.py) they guard against
# changes of this repository's results, not against a divergence from the reference that already existed.
# Whenever the reference sources are importable the tests also compare the live reference with the stored values.
RECORDED_RECORDS = os.path.join(GOLDEN, 'recorded_records.npz')
RECORDED_VALUES = os.path.join(GOLDEN, 'recorded_values.json')
_RECORD = os.environ.get('COBEL_RECORD_REFERENCE')
assert _RECORD in (None, 'reference', 'ours'), _RECORD
_INLINE = 256         # canonical forms longer than this (JSON characters) are stored as their SHA-256


def _reference_live():
    from oracle import ref_loader
    return ref_loader.available()


def _canonical(x):
    """JSON form of ``x`` under which equal forms mean ``==`` in Python: numbers as floats (0 == 0.0 == False),
    arrays with their dtype and shape, tuples apart from lists, dict items sorted (their order does not count)."""
    import json
    if hasattr(x, 'detach'):            # a torch tensor
        x = x.detach().cpu().numpy()
    if isinstance(x, np.ndarray):
        return {'ndarray': x.dtype.str, 'shape': list(x.shape), 'values': _canonical(x.ravel().tolist())}
    if isinstance(x, np.generic):
        x = x.item()
    if isinstance(x, (bool, int, float)):
        return float(x)
    if isinstance(x, dict):
        items = [(json.dumps(_canonical(k), sort_keys=True), _canonical(v)) for k, v in x.items()]
        return {'dict': sorted(items, key=lambda kv: kv[0])}
    if isinstance(x, tuple):
        return {'tuple': [_canonical(v) for v in x]}
    if isinstance(x, list):
        return [_canonical(v) for v in x]
    assert x is None or isinstance(x, str), type(x)
    return x


def _stored_form(x):
    """The canonical form of ``x`` if short, else its SHA-256 with the array dtype / shape or container length."""
    import hashlib
    import json
    c = _canonical(x)
    text = json.dumps(c, sort_keys=True)
    if len(text) <= _INLINE:
        return c
    out = {'sha256': hashlib.sha256(text.encode()).hexdigest()}
    if isinstance(c, dict) and 'ndarray' in c:
        out.update(ndarray=c['ndarray'], shape=c['shape'])
    elif isinstance(c, dict):
        out['len'] = len(next(iter(c.values())))
    elif isinstance(c, list):
        out['len'] = len(c)
    return out


def world_form(world):
    """A WorldDict as the reference builds it: without the product's successor table ``succ``, and with
    ``invalid_transitions`` as the sorted list of pairs (make_gridworld only tests membership)."""
    w = {k: v for k, v in world.items() if k != 'succ'}
    w['invalid_transitions'] = sorted((int(s), int(t)) for s, t in w['invalid_transitions'])
    return w


def check_stored(label, ours, live=None):
    """``ours`` equals the value recorded for ``label`` (see the provenance above); ``live()`` is the same call of the
    reference, compared with the recorded value when the reference sources are importable."""
    import json
    stored = json.load(open(RECORDED_VALUES)) if os.path.exists(RECORDED_VALUES) else {}
    if _RECORD:
        stored[label] = _stored_form(live() if _RECORD == 'reference' else ours)
        with open(RECORDED_VALUES, 'w') as f:         # one label per line
            f.write('{\n%s\n}\n' % ',\n'.join('%s: %s' % (json.dumps(k), json.dumps(v, sort_keys=True, separators=(',', ':')))
                                              for k, v in sorted(stored.items())))
        return
    assert label in stored, 'no recorded value for %s' % label
    for who, value in [('ours', ours)] + ([('live reference', live())] if live is not None and _reference_live() else []):
        got = json.loads(json.dumps(_stored_form(value)))
        assert got == stored[label], '%s: %s gives %.400s; recorded: %.400s' % (label, who, got, stored[label])


def check_stored_record(case, got, keys, live=None, rtol=None):
    """``got`` equals the arrays (e.g. trajectory, replay, tables, draws) recorded for ``case`` field by field over
    ``keys`` (see assert_equal_records and the provenance above); ``live()`` reruns the case in the reference."""
    stored = load_golden('recorded_records') if os.path.exists(RECORDED_RECORDS) else {}
    if _RECORD:
        rec = live() if _RECORD == 'reference' else got
        stored = {k: v for k, v in stored.items() if not k.startswith(case + '__')}
        stored.update({'%s__%s' % (case, k): np.asarray(rec[k]) for k in keys})
        np.savez_compressed(RECORDED_RECORDS, **stored)
        return
    want = {k[len(case) + 2:]: v for k, v in stored.items() if k.startswith(case + '__')}
    assert want, 'no recorded record for %s' % case
    assert_equal_records(got, want, keys, rtol=rtol, what=case)
    if live is not None and _reference_live():
        assert_equal_records(live(), want, keys, rtol=rtol, what='live reference, ' + case)


def make_world(name, tools=None):
    """WorldDict of a named case world, built with the product's builder by default."""
    if tools is None:
        from cobel_rl_b200.misc import gridworld_tools as tools
    h, w, kw = cases.world_args(name)
    kw = dict(kw)
    slip = kw.pop('slippery', None)
    world = tools.make_gridworld(h, w, **kw)
    return cases.make_slippery(world, slip) if slip else world


def make_topology(spec, tools=None):
    if tools is None:
        from cobel_rl_b200.misc import topology_tools as tools
    fn, args = spec
    return getattr(tools, fn)(*args)


def assert_equal_records(got, want, keys, rtol=None, what=''):
    for k in keys:
        g, w = np.asarray(got[k]), np.asarray(want[k])
        assert g.shape == w.shape, '%s %s: shape %s vs %s' % (what, k, g.shape, w.shape)
        if rtol is not None and k in rtol:
            # norm-wise relative tolerance: |got - want| <= rtol * max|want| (what LAPACK itself guarantees
            # for an inverse; tiny entries carry a larger element-wise relative error on both sides)
            err = np.abs(g - w).max() / np.abs(w).max()
            assert err <= rtol[k], '%s %s: norm-wise relative error %.3e > %.1e' % (what, k, err, rtol[k])
            np.testing.assert_allclose(g, w, rtol=1e-8, atol=rtol[k] * np.abs(w).max(), err_msg='%s %s' % (what, k))
        else:
            assert np.array_equal(g, w), '%s %s differs (max abs diff %s)' % (
                what, k, np.abs(g.astype(np.float64) - w.astype(np.float64)).max() if g.size else '')


def oracle_case(name, agent=None, golden=None):
    """Run the oracle restatement on a case; returns a record shaped like the goldens."""
    kind, wname, case_agent, args = cases.CASES[name]
    agent = case_agent if agent is None else agent
    a = dict(args)
    trials, steps = a.pop('trials'), a.pop('steps')
    valid_mask = a.pop('valid_mask', False)
    rng = tb.Draws(LazyStream(cases.SEED, agent), 1)      # env constructor consumed draw 0
    if kind in ('q_topo',):
        W = tb.compile_topology(*make_topology(wname))
    else:
        world = make_world(wname)
        W = tb.compile_gridworld(world)
    S, A = W['S'], W['A']
    if kind == 'dynaq':
        st = tb.dynaq_init(S, A)
        if valid_mask:
            st['action_mask'] = tb.valid_move_mask(W['succ'])
        out = tb.dynaq_train(W, st, rng, trials, steps, a.pop('batch'), **a).arrays()
        out.update(Q=st['Q'], Mr=st['Mr'], Ms=st['Ms'], Mt=st['Mt'], draws=rng.k)
        t = tb.tabular_test(W, st['Q'], rng, 5, steps, policy=('eps', 0.0),
                            action_mask=st['action_mask'] if a.get('mask_actions') else None).arrays()
        out.update({'test_' + k: v for k, v in t.items() if not k.startswith('replay')})
        out['draws_after_test'] = rng.k
    elif kind in ('q_grid', 'q_topo'):
        st = tb.q_init(S, A)
        out = tb.q_train(W, st, rng, trials, steps, a.pop('batch'), **a).arrays()
        out.update(Q=st['Q'], draws=rng.k, log_len=len(st['log']))
    elif kind == 'sr':
        st = tb.sr_init(S, A)
        if valid_mask:
            st['action_mask'] = tb.valid_move_mask(W['succ'])
        out = tb.sr_train(W, st, rng, trials, steps, **a).arrays()
        out.update(SR=st['SR'], rew=st['rew'], model=st['model'], draws=rng.k)
    elif kind == 'sfma':
        st = tb.sfma_init(S, A)
        if valid_mask:
            st['action_mask'] = tb.valid_move_mask(W['succ'])
        D = (golden if golden is not None else load_golden(name))['D']
        rk = {'recency': a.pop('recency')} if 'recency' in a else {}
        a['random_replay'] = a.pop('random_replay', False)
        out = tb.sfma_train(W, st, D, rng, trials, steps, a.pop('batch'), replay_kwargs=rk, **a).arrays()
        out.update(Q=st['Q'], Mr=st['Mr'], Ms=st['Ms'], Mt=st['Mt'], C=st['C'], T=st['T'], I=st['I'], draws=rng.k)
        if a.get('dynamic'):
            out.update(modes=np.array(st['modes'], dtype=np.int32), td=np.float64(st['td_acc']))
    elif kind == 'pma':
        st = tb.pma_init(tb.t0_from_succ(W['succ']), S, A)
        if valid_mask:
            st['action_mask'] = tb.valid_move_mask(W['succ'])
        if a.pop('prefill', False):
            st['Ms'][:] = W['succ']
            st['update_mask'] = tb.pma_compute_update_mask(st)
        cert = []
        out = tb.pma_train(W, st, rng, trials, steps, a.pop('batch'), cert=cert, **a).arrays()
        out.update(Q=st['Q'], Mr=st['Mr'], Ms=st['Ms'], Mt=st['Mt'], T=st['T'], SR=st['SR'],
                   update_mask=st['update_mask'], draws=rng.k, min_gap=min(cert))
    else:
        raise ValueError(kind)
    return out


# --------------------------------------------------------------------------- #
# CUDA side
# --------------------------------------------------------------------------- #

def policy_obj(spec, stream):
    from cobel_rl_b200 import policy as P
    kind, par = spec
    cls = {'eps': P.EpsilonGreedy, 'xeps': P.ExclusiveEpsilonGreedy, 'softmax': P.Softmax}[kind]
    return cls(par, rng=stream)


def unpack_run(res, i, A, succ, reward):
    """Record of local agent ``i`` from a RunResult with recorded traces."""
    ns = int(res['n_steps'][i])
    sa = res['step_sa'][i, :ns].cpu().numpy()
    s, a = sa // A, sa % A
    s2 = res['step_next'][i, :ns].cpu().numpy() if 'step_next' in res else np.asarray(succ)[s, a]
    nrep = int(res['n_replay'][i])
    rl = res['replay_len'][i].cpu().numpy()
    rl = rl[rl >= 0]
    return {
        'states': s.astype(np.int32), 'actions': a.astype(np.int32), 'next_states': s2.astype(np.int32),
        'rewards': np.asarray(reward, dtype=np.float64)[s2],
        'trial_steps': res['trial_steps'][i].cpu().numpy(), 'trial_reward': res['trial_reward'][i].cpu().numpy(),
        'replay': res['replay_idx'][i, :nrep].cpu().numpy(), 'replay_len': rl.astype(np.int32),
    }


def cuda_case(name, n_extra=2, device='cuda:0'):
    """Run a case of oracle/cases.py through the CUDA path.  The case's agent is local agent 0 of
    a batch of ``1 + n_extra`` agents (global ids agent .. agent+n_extra)."""
    import torch
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld, Topology
    from cobel_rl_b200 import agent as AG
    kind, wname, case_agent, args = cases.CASES[name]
    a = dict(args)
    trials, steps = a.pop('trials'), a.pop('steps')
    valid_mask = a.pop('valid_mask', False)
    stream = cb.BatchStream(1 + n_extra, seed=cases.SEED, device=device, agent_id_base=case_agent)
    if kind == 'q_topo':
        env = Topology(*make_topology(wname), rng=stream)
    else:
        env = Gridworld(make_world(wname), rng=stream)
    succ = env._succ.cpu().numpy()
    reward = env._reward.cpu().numpy()
    A = succ.shape[1]
    pol = policy_obj(a.pop('policy', ('eps', 0.1)), stream)
    if kind == 'dynaq':
        from cobel_rl_b200.memory import DynaQMemory
        mem = DynaQMemory(env.n_states, A, a.pop('mem_lr', 0.9), rng=stream)
        ag = AG.DynaQ(env.observation_space, env.action_space, pol, policy_obj(('eps', 0.0), stream),
                      a.pop('lr', 0.99), a.pop('gamma', 0.99), mem)
        ag.mask_actions = a.pop('mask_actions', False)
        ag.episodic_replay = a.pop('episodic_replay', False)
        if valid_mask:
            ag.action_mask = tb.valid_move_mask(succ)
        ag.record = True
        res = ag.train(env, trials, steps, a.pop('batch'), a.pop('no_replay', False))
        torch.cuda.synchronize()
        out = unpack_run(res, 0, A, succ, reward)
        out.update(Q=ag._Q[0].cpu().numpy(), Mr=mem._rewards[0].cpu().numpy(), Ms=mem._states[0].cpu().numpy(),
                   Mt=mem._terminals[0].cpu().numpy(), draws=int(stream.draw_count[0]))
        rt = ag.test(env, 5, steps)
        torch.cuda.synchronize()
        t = unpack_run(rt, 0, A, succ, reward)
        out.update({'test_' + k: v for k, v in t.items() if not k.startswith('replay')})
        out['draws_after_test'] = int(stream.draw_count[0])
        assert not a, 'unused case arguments %s' % a
        return out
    if kind in ('q_grid', 'q_topo'):
        ag = AG.QAgent(env.observation_space, env.action_space, pol, None, a.pop('lr', 0.9), a.pop('gamma', 0.8),
                       rng=stream)
        ag.record = True
        res = ag.train(env, trials, steps, a.pop('batch'))
        torch.cuda.synchronize()
        out = unpack_run(res, 0, A, succ, reward)
        out.update(Q=ag._Q[0].cpu().numpy(), draws=int(stream.draw_count[0]), log_len=int(ag._log_len[0]))
        assert not a, 'unused case arguments %s' % a
        return out
    if kind == 'sr':
        ag = AG.SR(env.observation_space, env.action_space, pol, None, a.pop('lr', 0.1), a.pop('gamma', 0.99))
        ag.mask_actions = a.pop('mask_actions', False)
        if valid_mask:
            ag.action_mask = tb.valid_move_mask(succ)
        ag.record = True
        res = ag.train(env, trials, steps)
        torch.cuda.synchronize()
        out = unpack_run(res, 0, A, succ, reward)
        out.update(SR=ag._SR[0].cpu().numpy(), rew=ag._rewards[0].cpu().numpy(), model=ag._model[0].cpu().numpy(),
                   draws=int(stream.draw_count[0]))
        assert not a, 'unused case arguments %s' % a
        return out
    if kind == 'sfma':
        from cobel_rl_b200.memory import SFMAMemory

        class _Metric:
            D = load_golden(name)['D']
        mem = SFMAMemory(_Metric(), env.n_states, A, learning_rate=a.pop('mem_lr', 0.9), rng=stream)
        mem.mode = a.pop('mode', 'default')
        mem.recency = a.pop('recency', False)
        ag = AG.SFMA(env.observation_space, env.action_space, pol, mem, None, a.pop('lr', 0.99), a.pop('gamma', 0.99),
                     rng=stream)
        ag.mask_actions = a.pop('mask_actions', False)
        ag.random = a.pop('random_replay', False)
        ag.dynamic = a.pop('dynamic', False)
        if valid_mask:
            ag.action_mask = tb.valid_move_mask(succ)
        ag.record = True
        res = ag.train(env, trials, steps, a.pop('batch'))
        torch.cuda.synchronize()
        out = unpack_run(res, 0, A, succ, reward)
        out.update(Q=ag._Q[0].cpu().numpy(), Mr=mem._rewards[0].cpu().numpy(), Ms=mem._states[0].cpu().numpy(),
                   Mt=mem._terminals[0].cpu().numpy(), C=mem._C[0].cpu().numpy(), T=mem._T[0].cpu().numpy(),
                   I=mem._I[0].cpu().numpy(), draws=int(stream.draw_count[0]), flags=int(res['flags'][0]))
        if ag.dynamic:      # golden 'modes' indexes ['reverse', 'default']; the kernel reports COBEL_SFMA_* ids
            rm = res['replay_mode'][0].cpu().numpy()
            assert set(np.unique(rm)) <= {0, 2}
            out.update(modes=np.where(rm == 2, 0, 1).astype(np.int32), td=np.float64(ag._td[0].item()))
        assert not a, 'unused case arguments %s' % a
        return out
    if kind == 'pma':
        from cobel_rl_b200.memory import PMAMemory
        world = make_world(wname)
        mem = PMAMemory(world['sas'], policy_obj(a.pop('mem_policy', ('eps', 0.1)), stream), a.pop('mem_lr', 0.9),
                        a.pop('lr_q', 0.9), a.pop('gamma_sr', 0.9), a.pop('gamma_q', 0.9), rng=stream)
        if a.pop('prefill', False):     # unit_tests/test_pma.py:69-73
            mem._states.copy_(env._succ.unsqueeze(0).expand_as(mem._states))
            mem.compute_update_mask()
        ag = AG.PMA(env.observation_space, env.action_space, pol, mem, None, a.pop('lr', 0.9), a.pop('gamma', 0.99))
        ag.mask_actions = a.pop('mask_actions', False)
        if valid_mask:
            ag.action_mask = tb.valid_move_mask(succ)
        ag.record = True
        res = ag.train(env, trials, steps, a.pop('batch'))
        torch.cuda.synchronize()
        out = unpack_run(res, 0, A, succ, reward)
        out.update(Q=ag._Q[0].cpu().numpy(), Mr=mem._rewards[0].cpu().numpy(), Ms=mem._states[0].cpu().numpy(),
                   Mt=mem._terminals[0].cpu().numpy(), T=mem._T[0].cpu().numpy(), SR=mem._SR[0].cpu().numpy(),
                   update_mask=mem._update_mask[0].cpu().numpy().astype(bool), draws=int(stream.draw_count[0]),
                   flags=int(res['flags'][0]), min_gap=float(mem._min_gap[0]))
        assert not a, 'unused case arguments %s' % a
        return out
    raise ValueError(kind)


# --------------------------------------------------------------------------- #
# full-size runs: the oracle on a SAMPLE of agents, one process per host core
# --------------------------------------------------------------------------- #

def sample_agents(n, per_group, k=32):
    """``k`` agent ids spread over the whole range: both ends, the last (possibly partial) CTA / warp group of
    ``per_group`` agents, and an even spread in between."""
    ids = {0, 1, n - 1, n - 2, max(n - per_group, 0), max(n - per_group - 1, 0), n // 2, n // 2 + 1}
    k = min(k, n)
    step = max(n // k, 1)
    i = 0
    while len(ids) < k:
        ids.add(min(i * step + (i * 7) % per_group, n - 1) if i < 2 * k else i - 2 * k)
        i += 1
    return sorted(ids)


def _oracle_sample_worker(job):
    kind, seed, g, cfg = job
    import numpy as np
    from oracle import tabular as tb
    from oracle.philox import LazyStream
    rng = tb.Draws(LazyStream(seed, g), 1)
    if kind == 'sr100':
        from cobel_rl_b200.misc.gridworld_tools import make_open_field
        world = make_open_field(100, 100, 0, 1, dense_sas=False)
        W = {'S': 10000, 'A': 4, 'succ': world['succ'], 'reward': world['rewards'].astype(np.float64),
             'terminal': world['terminals'].astype(np.uint8), 'starts': world['starting_states'].astype(np.int32)}
        st = tb.sr_init(10000, 4)
        rec = tb.sr_train(W, st, rng, cfg['trials'], cfg['steps']).arrays()
        nzr, nzc = np.nonzero(st['SR'])
        keep = nzr != nzc
        nzr, nzc = nzr[keep], nzc[keep]
        return {'trial_steps': rec['trial_steps'], 'draws': rng.k, 'SR_offdiag': (nzr, nzc, st['SR'][nzr, nzc]),
                'SR_diag': np.diag(st['SR']).copy()}
    if 'world_fn' in cfg:
        from cobel_rl_b200.misc import gridworld_tools
        world = getattr(gridworld_tools, cfg['world_fn'][0])(*cfg['world_fn'][1])
    else:
        world = make_world(cfg['world'])
    W = tb.compile_gridworld(world)
    S, A = W['S'], W['A']
    if kind == 'dynaq':
        st = tb.dynaq_init(S, A)
        rec = tb.dynaq_train(W, st, rng, cfg['trials'], cfg['steps'], cfg['batch']).arrays()
        return {'trial_steps': rec['trial_steps'], 'draws': rng.k, 'Q': st['Q'], 'Mr': st['Mr']}
    if kind == 'pma':
        st = tb.pma_init(tb.t0_from_succ(W['succ']), S, A)
        rec = tb.pma_train(W, st, rng, cfg['trials'], cfg['steps'], cfg['batch'], gamma_q=0.99, mask_actions=True).arrays()
        return {'trial_steps': rec['trial_steps'], 'draws': rng.k, 'Q': st['Q'], 'SR': st['SR'], 'T': st['T']}
    if kind == 'sfma':
        from cobel_rl_b200.memory.utils.metrics import DR
        D = DR(world['width'], world['height'], world['sas'], 0.9, world['invalid_transitions']).D
        st = tb.sfma_init(S, A)
        rec = tb.sfma_train(W, st, D, rng, cfg['trials'], cfg['steps'], cfg['batch'], mode=cfg.get('mode', 'default'),
                            mask_actions=True).arrays()
        return {'trial_steps': rec['trial_steps'], 'draws': rng.k, 'Q': st['Q'], 'C': st['C']}
    raise ValueError(kind)


def oracle_sample(kind, seed, agent_ids, **cfg):
    """{agent id: oracle result} for a sample of agents of a full-size run, computed on all host cores."""
    import multiprocessing as mp
    jobs = [(kind, seed, int(g), cfg) for g in agent_ids]
    procs = min(len(jobs), os.cpu_count() or 1, 16)
    with mp.get_context('spawn').Pool(procs) as pool:
        out = pool.map(_oracle_sample_worker, jobs, chunksize=1)
    return dict(zip([int(g) for g in agent_ids], out))


# ---- extended-precision reference for PMA's update_sr (SR = inv(I - gamma T) and the stationary need) -------------
# np.longdouble is the 80-bit format on x86-64 (eps 1.08e-19) and binary128 on aarch64 Linux (eps 1.9e-34); both are
# far enough below fp64 (eps 2.2e-16) that the reference's own error vanishes next to the kernels' gates.
LD = np.longdouble
EPS64 = float(np.finfo(np.float64).eps)


def _ld_check():
    assert np.finfo(LD).eps <= 1.1e-19, 'np.longdouble is not an extended format here: use mpmath for the reference'


def _lu_ld(A):
    """LU with partial pivoting in longdouble: (packed factors, row permutation)."""
    A = np.array(A, dtype=LD)
    S = A.shape[0]
    piv = np.arange(S)
    for k in range(S - 1):
        p = k + int(np.argmax(np.abs(A[k:, k])))
        if p != k:
            A[[k, p]] = A[[p, k]]
            piv[[k, p]] = piv[[p, k]]
        A[k + 1:, k] /= A[k, k]
        A[k + 1:, k + 1:] -= np.multiply.outer(A[k + 1:, k], A[k, k + 1:])
    return A, piv


def _lu_solve_ld(LU, piv, B):
    X = np.array(B, dtype=LD)[piv]
    S = LU.shape[0]
    for k in range(S):                         # L y = P b (unit diagonal)
        X[k + 1:] -= np.multiply.outer(LU[k + 1:, k], X[k])
    for k in range(S - 1, -1, -1):             # U x = y
        X[k] /= LU[k, k]
        X[:k] -= np.multiply.outer(LU[:k, k], X[k])
    return X


def ref_inverse(M):
    """inv(M) in longdouble: LU with partial pivoting, then two steps of iterative refinement whose residual
    I - M X is formed in longdouble."""
    _ld_check()
    M = np.array(M, dtype=LD)
    S = M.shape[0]
    I = np.eye(S, dtype=LD)
    LU, piv = _lu_ld(M)
    X = _lu_solve_ld(LU, piv, I)
    for _ in range(2):
        X += _lu_solve_ld(LU, piv, I - M @ X)
    return X


def ref_stationary(T):
    """Stationary distribution of the row-stochastic T by GTH elimination in longdouble, as |x| / ||x||_2 (what the
    kernels return).  GTH forms every quantity from the non-negative entries of T without a subtraction, so each
    entry -- the tiny ones of a nearly decoupled chain included -- has a small relative error."""
    _ld_check()
    P = np.array(T, dtype=LD)
    S = P.shape[0]
    for k in range(S - 1, 0, -1):
        s = P[k, :k].sum()
        P[:k, k] /= s
        P[:k, :k] += np.multiply.outer(P[:k, k], P[k, :k])
    x = np.zeros(S, dtype=LD)
    x[0] = 1
    for k in range(1, S):
        x[k] = x[:k] @ P[:k, k]
    x = np.abs(x)
    return x / np.sqrt((x * x).sum())


def nopivot_inverse(M):
    """inv(M) in fp64 by the kernels' own algorithm -- LU without pivoting, then L y = e_c and U x = y per column --
    in NumPy: the fp64 baseline of that elimination order, whose rounding errors differ from LAPACK's pivoted
    getrf / getri."""
    A = np.array(M, dtype=np.float64)
    S = A.shape[0]
    for k in range(S - 1):
        A[k + 1:, k] /= A[k, k]
        A[k + 1:, k + 1:] -= np.multiply.outer(A[k + 1:, k], A[k, k + 1:])
    X = np.eye(S)
    for k in range(S):
        X[k + 1:] -= np.multiply.outer(A[k + 1:, k], X[k])
    for k in range(S - 1, -1, -1):
        X[k] /= A[k, k]
        X[:k] -= np.multiply.outer(A[:k, k], X[k])
    return X


def kappa_inf(M, R):
    """kappa_inf(M) = ||M||_inf ||inv(M)||_inf with inv(M) = R."""
    return float(np.abs(np.asarray(M, dtype=LD)).sum(axis=1).max() * np.abs(R).sum(axis=1).max())


# Matrix generators (fixed seeds).  Every T is row-stochastic.
def _normalise(T):
    return T / T.sum(axis=1, keepdims=True)


def band_T(S, bw, seed):
    """Random T of half bandwidth bw with EVERY offset in [-bw, bw] non-zero (where it lies inside the matrix), its
    entries spread log-uniformly over 1e-8..1 before the rows are normalised."""
    rng = np.random.default_rng(seed)
    i, j = np.indices((S, S))
    T = np.where(np.abs(i - j) <= bw, 10.0 ** rng.uniform(-8, 0, (S, S)), 0.0)
    return _normalise(T)


def dense_T(S, seed):
    """Random dense T, entries log-uniform over 1e-8..1 before normalisation."""
    rng = np.random.default_rng(seed)
    return _normalise(10.0 ** rng.uniform(-8, 0, (S, S)))


def decoupled_T(S, seed, eps=1e-9):
    """Nearly decoupled chain: a block of states 0..m-1 leaks into the block m..S-1 only with probability `eps` (from
    state m-1), and every state of the second block returns to state 0 with probability 1/2.  The second block's
    stationary mass is about `eps` times the first's: the entries span more than 8 orders of magnitude.  S >= 2."""
    rng = np.random.default_rng(seed)
    m = max(1, S // 2)
    T = np.zeros((S, S))
    T[:m, :m] = _normalise(rng.uniform(0.1, 1.0, (m, m)))
    T[m - 1, :m] *= 1.0 - eps
    T[m - 1, m] = eps
    T[m:, m:] = 0.5 * _normalise(rng.uniform(0.1, 1.0, (S - m, S - m)))
    T[m:, 0] += 0.5
    return T


def reducible_T(S, seed, bw=None):
    """Two closed classes (states below S // 2 and the rest), no transition between them: no unique stationary
    distribution.  `bw`: each block is banded with that half width."""
    m = S // 2
    T = np.zeros((S, S))
    for lo, hi, k in ((0, m, 0), (m, S, 1)):
        n = hi - lo
        T[lo:hi, lo:hi] = dense_T(n, seed + k) if bw is None else band_T(n, bw, seed + k)
    return T
