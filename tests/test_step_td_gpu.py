"""GPU: ``last_run['step_td']``, the TD error of every step's online update recorded by the fused ``train()`` of Dyna-Q,
QAgent, SFMA and PMA.  For a spread of agents (the first, the last, those of a partial last CTA) every recorded entry
must have the bits of the online td of the oracle's training loop (oracle/tabular.py), the buffer must hold NaN behind
``n_steps``, and the trajectory must match the oracle.  Recording must not change the run: Q and the draw counts equal
those of the same run without ``record``."""
import inspect
from unittest import mock

import numpy as np
import pytest
import torch

from oracle import cases, tabular as tb
from oracle.philox import LazyStream
from helpers import load_golden, make_topology, make_world

pytestmark = pytest.mark.gpu


def _compile(world):
    """tb.compile_gridworld, also for worlds built without the dense ``sas`` (their successor table is ``succ``)."""
    if world['sas'] is not None:
        return tb.compile_gridworld(world)
    return {'sas': None, 'S': int(world['states']), 'A': 4, 'succ': np.asarray(world['succ'], dtype=np.int32),
            'reward': np.asarray(world['rewards'], dtype=np.float64).copy(),
            'terminal': np.asarray(world['terminals']).astype(np.uint8),
            'starts': np.asarray(world['starting_states']).astype(np.int32)}


class _TDRecord(tb.Record):
    """tb.Record that also keeps ``td``: the TD error of the online update of every recorded step."""

    def __init__(self):
        super().__init__()
        self.td, self.last_td = [], None

    def step(self, s, a, s2, r):
        super().step(s, a, s2, r)
        self.td.append(self.last_td)


def _oracle_train(fn, *args, **kw):
    """Run an oracle training loop (tb.dynaq_train, q_train, sfma_train, pma_train) and return its record with the
    online TD errors.  Dyna-Q, QAgent and SFMA update Q through tb._td_update: the last call before a recorded step
    is the step's online update (its replays follow the step).  PMA computes its online td inline; it is rebuilt
    from the row Q[s] that the step's action selection read, in pma_train's operation order, and must reproduce the
    update the oracle applied to Q[s, a] bit for bit."""
    rec = _TDRecord()
    td_update, select, store = tb._td_update, tb.select_action, tb.pma_store
    params = inspect.signature(fn).parameters
    lr, gamma = (kw.get(k, params[k].default) for k in ('lr', 'gamma'))
    row = {}

    def td_update_(*a, **k):
        rec.last_td = td_update(*a, **k)
        return rec.last_td

    def select_(policy, v, mask, rng):
        row['q'] = np.array(v, copy=True)
        return select(policy, v, mask, rng)

    def store_(st, s, a, r, s2, nt, *a_, **k_):
        Q, q = st['Q'], row['q']
        fv = np.amax(q if s2 == s else Q[s2]) * nt       # the update leaves Q[s2] as it was unless s2 == s
        rr = 0.0
        rr += r * (gamma ** 0)
        td = rr + fv * (gamma ** 1)
        td -= q[a]
        assert q[a] + lr * td == Q[s][a], "the rebuilt td does not reproduce the oracle's update"
        rec.last_td = td
        return store(st, s, a, r, s2, nt, *a_, **k_)

    with mock.patch.object(tb, '_td_update', td_update_), mock.patch.object(tb, 'select_action', select_), \
            mock.patch.object(tb, 'pma_store', store_):
        fn(*args, rec=rec, **kw)
    return rec


def _sample(n):
    return sorted({0, 1, n // 2, n - 2, n - 1})


def _check_td(res, i, rec, A, what):
    ns = int(res['n_steps'][i])
    assert ns == len(rec.td) > 0, '%s agent %d: %d steps, oracle %d' % (what, i, ns, len(rec.td))
    sa = res['step_sa'][i, :ns].cpu().numpy()
    assert np.array_equal(sa, np.array(rec.s) * A + np.array(rec.a)), '%s agent %d: trajectory' % (what, i)
    td = res['step_td'][i].cpu().numpy()
    want = np.array(rec.td, dtype=np.float64)
    bad = np.nonzero(td[:ns].view(np.uint64) != want.view(np.uint64))[0]
    assert bad.size == 0, '%s agent %d: step_td differs at step %d: %r vs oracle %r' % (
        what, i, bad[0], td[bad[0]], want[bad[0]])
    assert np.isnan(td[ns:]).all(), '%s agent %d: step_td behind n_steps is not NaN' % (what, i)


def _same_run(make, run, tables):
    """Train once with and once without ``record``; Q / tables and draw counts must agree; returns the recorded run."""
    out = []
    for record in (True, False):
        env, ag, stream = make()
        ag.record = record
        res = run(env, ag)
        torch.cuda.synchronize()
        assert ('step_td' in res) == record
        assert int(res['flags'].sum()) == 0, res['flags'].tolist()
        out.append((env, ag, stream, res, [t(ag).cpu().clone() for t in tables], stream.draw_count.cpu().clone()))
    (_, _, _, _, tab_r, dc_r), (_, _, _, _, tab_p, dc_p) = out
    for a, b in zip(tab_r, tab_p):
        assert torch.equal(a, b), 'recording changed the tables'
    assert torch.equal(dc_r, dc_p), 'recording changed the draw counts'
    return out[0][:4]


# ---- Dyna-Q --------------------------------------------------------------------------------------------------------

def _dynaq(world, n, seed, policy):
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
        return env, ag, stream
    return make


def _dynaq_oracle(world, seed, i, trials, steps, batch, policy):
    W = _compile(world)
    rng = tb.Draws(LazyStream(seed, i), 1)
    st = tb.dynaq_init(W['S'], W['A'])
    rec = _oracle_train(tb.dynaq_train, W, st, rng, trials, steps, batch, policy=policy, lr=0.99, gamma=0.99,
                        mem_lr=0.9)
    return rec, st, rng


@pytest.mark.parametrize('wname,policy', [('open5', ('eps', 0.1)), ('open5', ('softmax', 2.0)),
                                          ('slip5', ('eps', 0.1))])
def test_dynaq_5x5(wname, policy):
    """The 5x5 golden configuration (40 trials of 50 steps, batch 32); 37 agents: the last CTA of 4 holds one."""
    world, n, seed, trials, steps, batch = make_world(wname), 37, cases.SEED, 40, 50, 32
    env, ag, stream, res = _same_run(_dynaq(world, n, seed, policy), lambda e, a: a.train(e, trials, steps, batch),
                                     [lambda a: a._Q, lambda a: a.M._rewards])
    assert res['step_td'].dtype == torch.float64 and res['step_td'].shape == (n, trials * steps)
    for i in _sample(n):
        rec, st, rng = _dynaq_oracle(world, seed, i, trials, steps, batch, policy)
        _check_td(res, i, rec, 4, 'dynaq %s %s' % (wname, policy[0]))
        assert np.array_equal(ag._Q[i].cpu().numpy(), st['Q']) and int(stream.draw_count[i]) == rng.k


def test_dynaq_50x50_hbm():
    """2500 states: the tables exceed shared memory, dynaq_warp_kernel<A, false, true> keeps them in HBM."""
    from cobel_rl_b200.misc.gridworld_tools import make_open_field
    world, n, seed, trials, steps, batch = make_open_field(50, 50, 0, 1, dense_sas=False), 5, 77, 2, 300, 32
    env, ag, stream, res = _same_run(_dynaq(world, n, seed, ('eps', 0.1)),
                                     lambda e, a: a.train(e, trials, steps, batch), [lambda a: a._Q])
    for i in range(n):
        rec, st, rng = _dynaq_oracle(world, seed, i, trials, steps, batch, ('eps', 0.1))
        _check_td(res, i, rec, 4, 'dynaq 50x50')
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
    assert torch.equal(one['n_steps'], split['n_steps'])
    for i in range(n):
        ns = int(one['n_steps'][i])
        assert torch.equal(one['step_sa'][i, :ns], split['step_sa'][i, :ns])
        assert torch.equal(one['step_td'][i, :ns].view(torch.int64), split['step_td'][i, :ns].view(torch.int64))
        assert bool(split['step_td'][i, ns:].isnan().all())
    for i in (0, n - 1):
        rec, _, _ = _dynaq_oracle(world, seed, i, trials, steps, batch, ('eps', 0.2))
        _check_td(split, i, rec, 4, 'dynaq trials_per_launch')


def test_no_step_td_without_learning():
    """test() performs no update and records no step_td; train(no_replay=True) still learns and records it."""
    world, n, seed = make_world('open5'), 6, 5
    env, ag, stream = _dynaq(world, n, seed, ('eps', 0.1))()
    ag.record = True
    res = ag.train(env, 10, 20, 32, no_replay=True)
    assert 'step_td' in res
    W = _compile(world)
    for i in (0, n - 1):
        rng = tb.Draws(LazyStream(seed, i), 1)
        rec = _oracle_train(tb.dynaq_train, W, tb.dynaq_init(25, 4), rng, 10, 20, 32, no_replay=True)
        _check_td(res, i, rec, 4, 'dynaq no_replay')
    res = ag.test(env, 3, 20)
    assert 'step_td' not in res and 'step_sa' in res


def test_dynaq_hand_written_loop_matches_train():
    """The TD errors that DynaQ.update_q returns in a hand-written loop over the stand-alone methods are those
    that the fused train() records."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import DynaQ
    from cobel_rl_b200.memory import DynaQMemory
    from cobel_rl_b200.policy import EpsilonGreedy
    world, seed, trials, steps, batch = make_world('open5'), 1234, 6, 30, 32
    env, ag, stream = _dynaq(world, 1, seed, ('eps', 0.1))()
    ag.record = True
    fused = ag.train(env, trials, steps, batch)
    torch.cuda.synchronize()
    ns = int(fused['n_steps'][0])

    stream = cb.BatchStream(None, seed=seed, device='cuda:0')
    env = Gridworld(world, rng=stream)
    pol = EpsilonGreedy(0.1, rng=stream)
    mem = DynaQMemory(env.n_states, 4, 0.9, rng=stream)
    ag = DynaQ(env.observation_space, env.action_space, pol, None, 0.99, 0.99, mem)
    tds, sas = [], []
    for _ in range(trials):
        state, _info = env.reset()
        for _step in range(steps):
            action = pol.select_action(ag.Q[state], None)
            nxt, reward, end, _trunc, _info = env.step(action)
            exp = {'state': state, 'action': action, 'reward': reward, 'next_state': nxt, 'terminal': 1 - int(end)}
            mem.store(exp)
            tds.append(ag.update_q(exp)['td'])
            sas.append(int(state) * 4 + int(action))
            state = nxt
            ag.replay(batch)
            if end:
                break
    torch.cuda.synchronize()
    assert len(tds) == ns
    assert np.array_equal(np.array(sas), fused['step_sa'][0, :ns].cpu().numpy())
    assert np.array_equal(np.array(tds, dtype=np.float64).view(np.uint64),
                          fused['step_td'][0, :ns].cpu().numpy().view(np.uint64))


# ---- QAgent --------------------------------------------------------------------------------------------------------

def test_qagent_linear_track():
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Topology
    from cobel_rl_b200.agent import QAgent
    from cobel_rl_b200.policy import EpsilonGreedy
    spec = ('linear_track', (10, 2, 1.0, 20.0, 'right'))
    n, seed, trials, steps, batch = 13, cases.SEED, 25, 50, 8

    def make():
        stream = cb.BatchStream(n, seed=seed, device='cuda:0')
        env = Topology(*make_topology(spec), rng=stream)
        ag = QAgent(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream), None, 0.9, 0.8, rng=stream)
        return env, ag, stream
    env, ag, stream, res = _same_run(make, lambda e, a: a.train(e, trials, steps, batch), [lambda a: a._Q])
    W = tb.compile_topology(*make_topology(spec))
    for i in _sample(n):
        rng = tb.Draws(LazyStream(seed, i), 1)
        st = tb.q_init(W['S'], W['A'])
        rec = _oracle_train(tb.q_train, W, st, rng, trials, steps, batch, lr=0.9, gamma=0.8)
        _check_td(res, i, rec, W['A'], 'qagent track')
        assert np.array_equal(ag._Q[i].cpu().numpy(), st['Q']) and int(stream.draw_count[i]) == rng.k


# ---- SFMA ----------------------------------------------------------------------------------------------------------

def _sfma(world, D, S, n, seed, mem_opts, mask):
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
                  rng=stream)
        if mask:
            ag.mask_actions = True
            ag.action_mask = tb.valid_move_mask(_compile(world)['succ'])
        return env, ag, stream
    return make


def _sfma_check(world, D, n, seed, trials, steps, batch, mem_opts, mask, what, workspace=None):
    W = _compile(world)
    env, ag, stream, res = _same_run(_sfma(world, D, W['S'], n, seed, mem_opts, mask),
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
                            mask_actions=mask, replay_kwargs=rk, **kw)
        _check_td(res, i, rec, 4, what)
        assert np.array_equal(ag._Q[i].cpu().numpy(), st['Q']) and int(stream.draw_count[i]) == rng.k


def test_sfma_split_path():
    """Walled 5x5 world without per-step decay: the step kernel of the split path records step_td."""
    name = 'sfma_walls5_default'
    _sfma_check(make_world('walls5'), load_golden(name)['D'], 11, cases.SEED, 25, 50, 32, {'mode': 'default'}, True,
                'sfma split')


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

def _pma_check(world, n, seed, trials, steps, batch, band, what):
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
        ag = PMA(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream), mem)
        ag.mask_actions = True
        ag.action_mask = tb.valid_move_mask(W['succ'])
        if band < 0:
            mem.sr_band_max = -1
        assert mem.sr_band(env.transition_band)[0] == band
        return env, ag, stream
    env, ag, stream, res = _same_run(make, lambda e, a: a.train(e, trials, steps, batch), [lambda a: a._Q])
    for i in _sample(n):
        rng = tb.Draws(LazyStream(seed, i), 1)
        st = tb.pma_init(tb.t0_from_succ(W['succ']), W['S'], 4)
        st['action_mask'] = tb.valid_move_mask(W['succ'])
        rec = _oracle_train(tb.pma_train, W, st, rng, trials, steps, batch, gamma_q=0.99, mask_actions=True)
        _check_td(res, i, rec, 4, what)
        assert np.array_equal(ag._Q[i].cpu().numpy(), st['Q']) and int(stream.draw_count[i]) == rng.k


@pytest.mark.parametrize('band', [10, -1])
def test_pma_walls10(band):
    """10x10 walled world (config C3 shape) with the banded (band 10) and the dense (-1) update_sr."""
    _pma_check(make_world('walls10'), 7, 4242, 3, 60, 24, band, 'pma walls10 band %d' % band)


def test_pma_20x20_big():
    """400 states: pma_main_kernel<A, false, BIG>."""
    from cobel_rl_b200.misc import gridworld_tools as mg
    walls = [(5, 6), (6, 5), (25, 26), (26, 25), (45, 46), (46, 45), (208, 228), (228, 208), (209, 229), (229, 209)]
    world = mg.make_gridworld(20, 20, terminals=[19], rewards=np.array([[19, 10.0]]), goals=[19], starting_states=[210],
                              invalid_transitions=walls)
    _pma_check(world, 5, 2020, 2, 70, 16, 20, 'pma 20x20')
