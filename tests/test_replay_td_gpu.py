"""GPU: ``last_run['replay_td']``, the TD error of every replayed update recorded by the fused ``train()`` of Dyna-Q,
QAgent, SFMA and PMA.  For a spread of agents (the first, the last, those of a partial last CTA) every entry up to
``n_replay`` must have the bits of the td that the oracle's replay (oracle/tabular.py) computes for the same replayed
experience, aligned with ``replay_idx``, and the buffer must hold NaN behind ``n_replay``.  PMA records, per performed
update, the td of the sequence element that ``replay_idx`` names, NaN where the n-step update aborts.  Recording must
not change the run: Q, the draw counts, ``replay_idx`` and ``step_td`` equal those of the same recorded run whose
``replay_td`` is left NULL."""
from unittest import mock

import numpy as np
import pytest
import torch

from oracle import cases, tabular as tb
from oracle.philox import LazyStream
from helpers import load_golden, make_topology, make_world

pytestmark = pytest.mark.gpu

NAN = float('nan')


def _compile(world):
    """tb.compile_gridworld, also for worlds built without the dense ``sas`` (their successor table is ``succ``)."""
    if world['sas'] is not None:
        return tb.compile_gridworld(world)
    return {'sas': None, 'S': int(world['states']), 'A': 4, 'succ': np.asarray(world['succ'], dtype=np.int32),
            'reward': np.asarray(world['rewards'], dtype=np.float64).copy(),
            'terminal': np.asarray(world['terminals']).astype(np.uint8),
            'starts': np.asarray(world['starting_states']).astype(np.int32)}


# ---- the oracle's replayed TD errors -------------------------------------------------------------------------------

class _Replays(list):
    """``Record.replay`` that, whenever a replay call logs its experiences, takes the TD errors of the updates that the
    call applied (one per experience; none for a replay that updates nothing, which gets NaN)."""

    def __init__(self, rec):
        super().__init__()
        self.rec = rec

    def extend(self, idx):
        idx = list(idx)
        tds = self.rec.pending
        assert len(tds) in (0, len(idx)), 'a replay call of %d experiences applied %d updates' % (len(idx), len(tds))
        self.rec.replay_td.extend(tds if tds else [NAN] * len(idx))
        self.rec.pending = []
        super().extend(idx)


class _ReplayTDRecord(tb.Record):
    def __init__(self):
        super().__init__()
        self.replay = _Replays(self)
        self.replay_td, self.pending = [], []
        self.loops = 0             # PMA: applied sequences that revisit a state

    def step(self, s, a, s2, r):
        super().step(s, a, s2, r)
        self.pending = []          # the online update of the step is not a replayed one


class _Writes(np.ndarray):
    """View of a Q table that logs (old, new) of every entry written through it or through the row views it hands out
    (the oracle writes ``Qx[s][a] += ...``)."""

    def __array_finalize__(self, obj):
        self.log = getattr(obj, 'log', None)

    def __setitem__(self, key, value):
        old = np.ndarray.__getitem__(self, key)
        np.ndarray.__setitem__(self, key, value)
        if self.log is not None:
            self.log.append((old, np.ndarray.__getitem__(self, key)))


def _oracle_train(fn, *args, **kw):
    """Run an oracle training loop with its record capturing the replayed TD errors.  Dyna-Q, QAgent and SFMA replay
    through tb._td_update; PMA applies each performed update through tb.pma_update_q_sequence, whose last element's
    td is rebuilt here and must reproduce the update the oracle applied bit for bit."""
    rec = _ReplayTDRecord()
    td_update, seq_update = tb._td_update, tb.pma_update_q_sequence

    def td_update_(*a, **k):
        td = td_update(*a, **k)
        rec.pending.append(td)
        return td

    def seq_update_(st, Qx, seq, lr_q, gamma_q):
        # tb.pma_update_q_sequence applies the elements in order and writes nothing when it aborts (with n >= 2, at
        # the first element, if any element's M.terminals is 0).  The td of the last element is rebuilt in the
        # oracle's operation order from the Q value that its update read, the one logged last, also when a sequence
        # with loops has updated that entry before.
        S = Qx.shape[0]
        ls, la = seq[-1] % S, seq[-1] // S
        fv = np.amax(Qx[int(st['Ms'][ls, la])]) * st['Mt'][ls, la]
        tracked = Qx.view(_Writes)
        tracked.log = log = []
        seq_update(st, tracked, seq, lr_q, gamma_q)
        if not log:
            assert len(seq) >= 2 and any(st['Mt'][k % S, k // S] == 0 for k in seq)
            td = NAN
        else:
            assert len(log) == len(seq)
            q, qn = log[-1]
            r = 0.0
            r += st['Mr'][ls, la] * (gamma_q ** 0)
            td = r + fv * (gamma_q ** 1)
            td -= q
            assert q + lr_q * td == qn, "the rebuilt td does not reproduce the oracle's update"
        rec.pending.append(td)
        rec.loops += len({k % S for k in seq}) < len(seq)
        return Qx

    with mock.patch.object(tb, '_td_update', td_update_), mock.patch.object(tb, 'pma_update_q_sequence', seq_update_):
        fn(*args, rec=rec, **kw)
    return rec


# ---- checks --------------------------------------------------------------------------------------------------------

def _sample(n):
    return sorted({0, 1, n // 2, n - 2, n - 1})


def _same_bits(a, b):
    """Equal doubles bit for bit, any NaN equal to any NaN."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return (a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))


def _check_replay_td(res, i, rec, what):
    nr = int(res['n_replay'][i])
    assert nr == len(rec.replay) == len(rec.replay_td) > 0, '%s agent %d: %d replayed, oracle %d' % (
        what, i, nr, len(rec.replay))
    assert np.array_equal(res['replay_idx'][i, :nr].cpu().numpy(), np.array(rec.replay)), '%s agent %d: replay_idx' % (
        what, i)
    td = res['replay_td'][i].cpu().numpy()
    want = np.array(rec.replay_td, dtype=np.float64)
    bad = np.nonzero(~_same_bits(td[:nr], want))[0]
    assert bad.size == 0, '%s agent %d: replay_td differs at entry %d of %d: %r vs oracle %r' % (
        what, i, bad[0], nr, td[bad[0]], want[bad[0]])
    assert np.isnan(td[nr:]).all(), '%s agent %d: replay_td behind n_replay is not NaN' % (what, i)
    return int(np.isnan(want).sum())


def _without_replay_td():
    """Patch that keeps recording on but leaves CobelTrace.replay_td NULL."""
    from cobel_rl_b200.agent.agent import Agent
    make = Agent._make_trace

    def make_trace(self, *a, **k):
        k['replay_td'] = False
        return make(self, *a, **k)
    return mock.patch.object(Agent, '_make_trace', make_trace)


def _same_run(make, run, tables):
    """Train once recording replay_td and once recording everything else; the tables, draw counts and every other
    recorded buffer must agree.  Returns the run with replay_td."""
    out = []
    for with_td in (True, False):
        env, ag, stream = make()
        ag.record = True
        if with_td:
            res = run(env, ag)
        else:
            with _without_replay_td():
                res = run(env, ag)
        torch.cuda.synchronize()
        assert ('replay_td' in res) == with_td
        assert int(res['flags'].sum()) == 0, res['flags'].tolist()
        out.append((env, ag, stream, res, [t(ag).cpu().clone() for t in tables], stream.draw_count.cpu().clone()))
    (_, _, _, res_r, tab_r, dc_r), (_, _, _, res_p, tab_p, dc_p) = out
    for a, b in zip(tab_r, tab_p):
        assert torch.equal(a, b), 'recording replay_td changed the tables'
    assert torch.equal(dc_r, dc_p), 'recording replay_td changed the draw counts'
    for k in res_p:
        a, b = res_r[k], res_p[k]
        if a.dtype == torch.float64:
            a, b = a.view(torch.int64), b.view(torch.int64)
        assert torch.equal(a, b), 'recording replay_td changed %s' % k
    assert res_r['replay_td'].dtype == torch.float64 and res_r['replay_td'].shape == res_r['replay_idx'].shape
    return out[0][:4]


# ---- Dyna-Q --------------------------------------------------------------------------------------------------------

def _dynaq(world, n, seed, policy, mask=False, episodic=False):
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import DynaQ
    from cobel_rl_b200.memory import DynaQMemory
    from helpers import policy_obj

    def make():
        stream = cb.BatchStream(n, seed=seed, device='cuda:0')
        env = Gridworld(world, rng=stream)
        mem = DynaQMemory(env.n_states, 4, 0.9, rng=stream)
        ag = DynaQ(env.observation_space, env.action_space, policy_obj(policy, stream), None, 0.99, 0.99, mem)
        if mask:
            ag.mask_actions = True
            ag.action_mask = tb.valid_move_mask(_compile(world)['succ'])
        ag.episodic_replay = episodic
        return env, ag, stream
    return make


def _dynaq_oracle(world, seed, i, trials, steps, batch, policy, mask=False, episodic=False):
    W = _compile(world)
    rng = tb.Draws(LazyStream(seed, i), 1)
    st = tb.dynaq_init(W['S'], W['A'])
    if mask:
        st['action_mask'] = tb.valid_move_mask(W['succ'])
    rec = _oracle_train(tb.dynaq_train, W, st, rng, trials, steps, batch, policy=policy, lr=0.99, gamma=0.99,
                        mem_lr=0.9, mask_actions=mask, episodic_replay=episodic)
    return rec, st, rng


@pytest.mark.parametrize('wname,policy,mask,episodic', [
    ('open5', ('eps', 0.1), False, False), ('open5', ('softmax', 2.0), False, False),
    ('walls5', ('eps', 0.1), True, False), ('open5', ('eps', 0.1), False, True), ('slip5', ('eps', 0.1), False, False)])
def test_dynaq_5x5(wname, policy, mask, episodic):
    """The 5x5 golden configuration (40 trials of 50 steps, batch 32); 37 agents: the last CTA of 4 holds one.  The
    variants: softmax, an action mask, one replay per trial (episodic_replay), a stochastic world."""
    world, n, seed, trials, steps, batch = make_world(wname), 37, cases.SEED, 40, 50, 32
    env, ag, stream, res = _same_run(_dynaq(world, n, seed, policy, mask, episodic),
                                     lambda e, a: a.train(e, trials, steps, batch),
                                     [lambda a: a._Q, lambda a: a.M._rewards])
    for i in _sample(n):
        rec, st, rng = _dynaq_oracle(world, seed, i, trials, steps, batch, policy, mask, episodic)
        _check_replay_td(res, i, rec, 'dynaq %s %s mask %d episodic %d' % (wname, policy[0], mask, episodic))
        assert np.array_equal(ag._Q[i].cpu().numpy(), st['Q']) and int(stream.draw_count[i]) == rng.k


def test_dynaq_50x50_hbm():
    """2500 states: the tables exceed shared memory, dynaq_warp_kernel<A, false, true> keeps them in HBM."""
    from cobel_rl_b200.misc.gridworld_tools import make_open_field
    world, n, seed, trials, steps, batch = make_open_field(50, 50, 0, 1, dense_sas=False), 5, 77, 2, 300, 32
    env, ag, stream, res = _same_run(_dynaq(world, n, seed, ('eps', 0.1)),
                                     lambda e, a: a.train(e, trials, steps, batch), [lambda a: a._Q])
    for i in range(n):
        rec, st, rng = _dynaq_oracle(world, seed, i, trials, steps, batch, ('eps', 0.1))
        _check_replay_td(res, i, rec, 'dynaq 50x50')
        assert np.array_equal(ag._Q[i].cpu().numpy(), st['Q'])


def test_dynaq_trials_per_launch_equals_one_launch():
    world, n, seed, trials, steps, batch = make_world('open5'), 9, 31, 13, 30, 32
    runs = []
    for per_launch in (None, 4):
        env, ag, stream = _dynaq(world, n, seed, ('eps', 0.2))()
        ag.record = True
        ag.trials_per_launch = per_launch
        runs.append(ag.train(env, trials, steps, batch))
    torch.cuda.synchronize()
    one, split = runs
    assert torch.equal(one['n_replay'], split['n_replay'])
    for i in range(n):
        nr = int(one['n_replay'][i])
        assert torch.equal(one['replay_idx'][i, :nr], split['replay_idx'][i, :nr])
        assert torch.equal(one['replay_td'][i, :nr].view(torch.int64), split['replay_td'][i, :nr].view(torch.int64))
        assert bool(split['replay_td'][i, nr:].isnan().all())
    for i in (0, n - 1):
        rec, _, _ = _dynaq_oracle(world, seed, i, trials, steps, batch, ('eps', 0.2))
        _check_replay_td(split, i, rec, 'dynaq trials_per_launch')


# ---- QAgent --------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize('batch', [8, 0])
def test_qagent_linear_track(batch):
    """Replays over the experience log; batch 0 replays nothing and leaves the buffer NaN."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Topology
    from cobel_rl_b200.agent import QAgent
    from cobel_rl_b200.policy import EpsilonGreedy
    spec = ('linear_track', (10, 2, 1.0, 20.0, 'right'))
    n, seed, trials, steps = 13, cases.SEED, 25, 50

    def make():
        stream = cb.BatchStream(n, seed=seed, device='cuda:0')
        env = Topology(*make_topology(spec), rng=stream)
        ag = QAgent(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream), None, 0.9, 0.8, rng=stream)
        return env, ag, stream
    env, ag, stream, res = _same_run(make, lambda e, a: a.train(e, trials, steps, batch), [lambda a: a._Q])
    if batch == 0:
        assert int(res['n_replay'].sum()) == 0 and bool(res['replay_td'].isnan().all())
        return
    W = tb.compile_topology(*make_topology(spec))
    for i in _sample(n):
        rng = tb.Draws(LazyStream(seed, i), 1)
        st = tb.q_init(W['S'], W['A'])
        rec = _oracle_train(tb.q_train, W, st, rng, trials, steps, batch, lr=0.9, gamma=0.8)
        _check_replay_td(res, i, rec, 'qagent track')
        assert np.array_equal(ag._Q[i].cpu().numpy(), st['Q']) and int(stream.draw_count[i]) == rng.k


# ---- SFMA ----------------------------------------------------------------------------------------------------------

def _sfma(world, D, S, n, seed, mem_opts, mask, callbacks=None, start_replay=False, random=False):
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SFMA
    from cobel_rl_b200.memory import SFMAMemory
    from cobel_rl_b200.policy import EpsilonGreedy

    class _Metric:
        pass
    _Metric.D = D

    def make():
        stream = cb.BatchStream(n, seed=seed, device='cuda:0')
        env = Gridworld(world, rng=stream)
        mem = SFMAMemory(_Metric(), S, 4, learning_rate=0.9, rng=stream)
        for k, v in mem_opts.items():
            assert hasattr(mem, k), k
            setattr(mem, k, v)
        ag = SFMA(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream), mem, None, 0.99, 0.99,
                  custom_callbacks=callbacks, rng=stream)
        ag.start_replay = start_replay
        ag.random = random
        if mask:
            ag.mask_actions = True
            ag.action_mask = tb.valid_move_mask(_compile(world)['succ'])
        return env, ag, stream
    return make


def _sfma_check(world, D, n, seed, trials, steps, batch, mem_opts, mask, what, workspace=None, start_replay=False,
                random=False):
    W = _compile(world)
    env, ag, stream, res = _same_run(_sfma(world, D, W['S'], n, seed, mem_opts, mask, start_replay=start_replay,
                                           random=random),
                                     lambda e, a: a.train(e, trials, steps, batch),
                                     [lambda a: a._Q, lambda a: a.M._C])
    if workspace is not None:
        assert (ag.M._workspace is not None) == workspace
    for i in _sample(n):
        rng = tb.Draws(LazyStream(seed, i), 1)
        st = tb.sfma_init(W['S'], 4)
        if mask:
            st['action_mask'] = tb.valid_move_mask(W['succ'])
        kw = {k: v for k, v in mem_opts.items() if k == 'decay_strength'}
        rk = {k: v for k, v in mem_opts.items() if k == 'recency'}
        rec = _oracle_train(tb.sfma_train, W, st, D, rng, trials, steps, batch, mode=mem_opts.get('mode', 'default'),
                            mask_actions=mask, replay_kwargs=rk, start_replay=start_replay, random_replay=random, **kw)
        nan = _check_replay_td(res, i, rec, what)
        assert start_replay or nan == 0
        assert np.array_equal(ag._Q[i].cpu().numpy(), st['Q']) and int(stream.draw_count[i]) == rng.k


@pytest.mark.parametrize('mode', ['default', 'reverse'])
def test_sfma_split_path(mode):
    """Walled 5x5 world with an action mask (the replay's maximum is the masked one), no per-step decay: the replay
    kernel of the split path records replay_td."""
    name = 'sfma_walls5_%s' % mode
    _sfma_check(make_world('walls5'), load_golden(name)['D'], 11, cases.SEED, 25, 50, 32, {'mode': mode}, True,
                'sfma split %s' % mode)


def test_sfma_split_path_start_replay():
    """The trace-only replay at trial start updates nothing: its entries stay NaN, the replays at trial end record."""
    name = 'sfma_walls5_default'
    _sfma_check(make_world('walls5'), load_golden(name)['D'], 6, 17, 12, 50, 16, {'mode': 'default'}, True,
                'sfma split start_replay', start_replay=True)


@pytest.mark.parametrize('decay', [1.0, 0.9])
def test_sfma_random_replay(decay):
    """agent.random: uniform batches over the unmasked experiences, on the split path (decay_strength 1) and in the
    fused kernel (0.9)."""
    name = 'sfma_walls5_random'
    _sfma_check(make_world('walls5'), load_golden(name)['D'], 11, 321, 20, 50, 32,
                {'mode': 'default', 'decay_strength': decay}, True, 'sfma random decay %g' % decay,
                workspace=False if decay != 1.0 else None, random=True)


def test_sfma_fused_decay_strength():
    """decay_strength != 1 needs the fused kernel sfma_kernel<A, MODS, false>."""
    name = 'sfma_walls5_default'
    _sfma_check(make_world('walls5'), load_golden(name)['D'], 11, 99, 20, 50, 32,
                {'mode': 'default', 'decay_strength': 0.9}, True, 'sfma fused decay_strength', workspace=False)


def test_sfma_recency_50x50_workspace():
    """recency on 2500 states: the fused kernel with its tables in the global workspace (sfma_kernel<A, MODS, true>)."""
    from cobel_rl_b200.misc.gridworld_tools import make_open_field
    from cobel_rl_b200.memory.utils.metrics import Euclidean
    world = make_open_field(50, 50, 0, 1, dense_sas=False)
    _sfma_check(world, Euclidean(50, 50).D, 3, 4001, 3, 80, 32, {'mode': 'default', 'recency': True}, False,
                'sfma 50x50 recency', workspace=True)


# ---- PMA -----------------------------------------------------------------------------------------------------------

def _pma(world, n, seed, band, callbacks=None, opts=None):
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import PMA
    from cobel_rl_b200.memory import PMAMemory
    from cobel_rl_b200.policy import EpsilonGreedy
    W = _compile(world)

    def make():
        stream = cb.BatchStream(n, seed=seed, device='cuda:0')
        env = Gridworld(world, rng=stream)
        mem = PMAMemory(world['sas'], EpsilonGreedy(0.1, rng=stream), 0.9, 0.9, 0.9, 0.99, rng=stream)
        ag = PMA(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream), mem,
                 custom_callbacks=callbacks)
        ag.mask_actions = True
        ag.action_mask = tb.valid_move_mask(W['succ'])
        for k, v in (opts or {}).items():
            assert hasattr(mem, k), k
            setattr(mem, k, v)
        if band < 0:
            mem.sr_band_max = -1
        assert mem.sr_band(env.transition_band)[0] == band
        return env, ag, stream
    return make


def _pma_check(world, n, seed, trials, steps, batch, band, what, opts=None):
    """Returns the numbers of aborted n-step updates and of applied sequences with loops among the sampled agents."""
    W = _compile(world)
    env, ag, stream, res = _same_run(_pma(world, n, seed, band, opts=opts), lambda e, a: a.train(e, trials, steps, batch),
                                     [lambda a: a._Q])
    aborted = loops = 0
    for i in _sample(n):
        rng = tb.Draws(LazyStream(seed, i), 1)
        st = tb.pma_init(tb.t0_from_succ(W['succ']), W['S'], 4)
        st['action_mask'] = tb.valid_move_mask(W['succ'])
        rec = _oracle_train(tb.pma_train, W, st, rng, trials, steps, batch, gamma_q=0.99, mask_actions=True,
                            replay_kwargs=dict(opts or {}))
        aborted += _check_replay_td(res, i, rec, what)
        loops += rec.loops
        assert np.array_equal(ag._Q[i].cpu().numpy(), st['Q']) and int(stream.draw_count[i]) == rng.k
    return aborted, loops


@pytest.mark.parametrize('band', [10, -1])
def test_pma_walls10(band):
    """10x10 walled world (config C3 shape) with the banded (band 10) and the dense (-1) update_sr.  Its replays extend
    sequences into the goal, whose never-experienced transitions abort the n-step update: those entries are NaN in the
    oracle and in the recorded buffer."""
    aborted, _ = _pma_check(make_world('walls10'), 7, 4242, 3, 60, 24, band, 'pma walls10 band %d' % band)
    assert aborted > 0, 'the case is meant to contain aborted n-step updates'


def test_pma_walls10_allow_loops():
    """M.allow_loops: a sequence may revisit a state, and lane 0 applies its elements in order; the recorded td is the
    one of the last element's update, after the earlier elements have changed its entry where the sequence loops."""
    _, loops = _pma_check(make_world('walls10'), 7, 4242, 3, 60, 24, 10, 'pma walls10 allow_loops',
                          opts={'allow_loops': True})
    assert loops > 0, 'the case is meant to apply sequences with loops'


def test_pma_20x20_big():
    """400 states: pma_main_kernel<A, false, BIG>."""
    from cobel_rl_b200.misc import gridworld_tools as mg
    walls = [(5, 6), (6, 5), (25, 26), (26, 25), (45, 46), (46, 45), (208, 228), (228, 208), (209, 229), (229, 209)]
    world = mg.make_gridworld(20, 20, terminals=[19], rewards=np.array([[19, 10.0]]), goals=[19], starting_states=[210],
                              invalid_transitions=walls)
    _pma_check(world, 5, 2020, 2, 70, 16, 20, 'pma 20x20')


def test_pma_trials_per_launch_equals_one_launch():
    world, n, seed, trials, steps, batch = make_world('walls10'), 5, 4242, 5, 60, 24
    runs = []
    for per_launch in (None, 2):
        env, ag, stream = _pma(world, n, seed, 10)()
        ag.record = True
        ag.trials_per_launch = per_launch
        runs.append(ag.train(env, trials, steps, batch))
    torch.cuda.synchronize()
    one, split = runs
    assert torch.equal(one['n_replay'], split['n_replay'])
    for i in range(n):
        nr = int(one['n_replay'][i])
        assert torch.equal(one['replay_idx'][i, :nr], split['replay_idx'][i, :nr])
        assert bool(_same_bits(one['replay_td'][i, :nr].cpu().numpy(), split['replay_td'][i, :nr].cpu().numpy()).all())
        assert bool(split['replay_td'][i, nr:].isnan().all())


# ---- callbacks and the calls that record nothing -------------------------------------------------------------------

def _replay_logs_match(res, got, what):
    """logs['replay']['td'] of every on_replay_end call equals the slice of replay_td that the call's experiences
    occupy, NaN where index is -1."""
    n = res['n_replay'].shape[0]
    offset = torch.zeros(n, dtype=torch.long, device=res['n_replay'].device)
    for r in got:
        idx, td, ln = r['index'], r['td'], r['length'].long()
        assert td.dtype == torch.float64 and td.shape == idx.shape
        assert bool(td[idx < 0].isnan().all()), what
        for i in range(n):
            k = int(ln[i])
            want = res['replay_td'][i, int(offset[i]):int(offset[i]) + k].cpu().numpy()
            assert bool(_same_bits(td[i, :k].cpu().numpy(), want).all()), '%s agent %d' % (what, i)
        offset += ln
    assert torch.equal(offset, res['n_replay'].long()), what


def test_replay_callbacks_carry_td():
    world = make_world('walls10')
    got = []
    cbs = {'on_replay_end': [lambda logs: got.append(logs['replay'])]}
    env, ag, stream = _pma(world, 5, 4242, 10, callbacks=cbs)()
    ag.record = True
    res = ag.train(env, 4, 60, 24)
    torch.cuda.synchronize()
    assert len(got) == 8
    _replay_logs_match(res, got, 'pma')
    assert bool(res['replay_td'][:, :int(res['n_replay'].min())].isnan().any()), 'expected aborted updates'

    W = _compile(make_world('walls5'))
    got.clear()
    make = _sfma(make_world('walls5'), load_golden('sfma_walls5_default')['D'], W['S'], 4, 5, {'mode': 'default'},
                 True, callbacks=cbs, start_replay=True)
    env, ag, stream = make()
    ag.record = True
    res = ag.train(env, 5, 40, 16)
    torch.cuda.synchronize()
    assert len(got) == 10
    _replay_logs_match(res, got, 'sfma')
    assert bool(got[0]['td'].isnan().all()) and not bool(got[1]['td'][got[1]['index'] >= 0].isnan().any())


def test_no_replay_td_without_replayed_updates():
    """test() and train(no_replay=True) allocate no replay_td, and nothing else in the run changes for it."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Topology
    from cobel_rl_b200.agent import QAgent
    from cobel_rl_b200.policy import EpsilonGreedy
    world = make_world('walls5')
    W = _compile(world)
    D = load_golden('sfma_walls5_default')['D']
    makers = {'dynaq': _dynaq(world, 6, 5, ('eps', 0.1)), 'pma': _pma(make_world('walls10'), 3, 5, 10),
              'sfma': _sfma(world, D, W['S'], 4, 5, {'mode': 'default'}, True, start_replay=True)}
    for name, make in makers.items():
        env, ag, stream = make()
        ag.record = True
        res = ag.train(env, 3, 20, 8, no_replay=True)
        assert 'replay_td' not in res and 'step_td' in res, name
        res = ag.test(env, 2, 20)
        assert 'replay_td' not in res and 'step_sa' in res, name
    spec = ('linear_track', (10, 2, 1.0, 20.0, 'right'))
    stream = cb.BatchStream(3, seed=5, device='cuda:0')
    env = Topology(*make_topology(spec), rng=stream)
    ag = QAgent(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream), None, 0.9, 0.8, rng=stream)
    ag.record = True
    assert 'replay_td' in ag.train(env, 2, 20, 4)
    res = ag.test(env, 2, 20)
    assert 'replay_td' not in res and 'step_sa' in res
    torch.cuda.synchronize()
