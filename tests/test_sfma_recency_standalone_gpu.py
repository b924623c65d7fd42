"""GPU: SFMA's stand-alone replay with the recency option (the priority C * D * (1 - I) weighted by M.T, memory/sfma.py:311):
the reference's train loop written by hand over store / update_q / replay / M.T.fill(0) lands on the golden of the
fused train(), and SFMAMemory.replay matches the oracle (oracle/tabular.py: sfma_memory_replay) on worlds whose tables
fit in shared memory and on worlds whose tables do not."""
import numpy as np
import pytest
import torch

from oracle import cases, tabular as tb
from oracle.philox import LazyStream
from helpers import KEYS, assert_equal_records, load_golden, make_world

pytestmark = pytest.mark.gpu


def test_hand_written_loop_with_recency_matches_golden():
    """agent/sfma.py:266-327 one call at a time on a single-agent stream: sweeping mode, action mask, recency."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SFMA
    from cobel_rl_b200.memory import SFMAMemory
    from cobel_rl_b200.policy import EpsilonGreedy
    name = 'sfma_walls5_sweeping_recency'
    kind, wname, case_agent, a = cases.CASES[name]
    assert a['recency'] and a['mode'] == 'sweeping' and a['mask_actions']
    stream = cb.BatchStream(None, seed=cases.SEED, device='cuda:0', agent_id_base=case_agent)
    env = Gridworld(make_world(wname), rng=stream)
    pol = EpsilonGreedy(0.1, rng=stream)
    golden = load_golden(name)

    class _Metric:
        D = golden['D']
    mem = SFMAMemory(_Metric(), env.n_states, 4, learning_rate=0.9, rng=stream)
    mem.mode, mem.recency = a['mode'], True
    ag = SFMA(env.observation_space, env.action_space, pol, mem, None, 0.99, 0.99, rng=stream)
    ag.mask_actions = True
    mask = ag.action_mask
    S = env.n_states
    got = {k: [] for k in ('states', 'actions', 'next_states', 'rewards', 'trial_steps', 'trial_reward', 'replay',
                           'replay_len')}
    for _ in range(a['trials']):
        state, _info = env.reset()
        total, step, last = 0.0, 0, None
        for step in range(a['steps']):
            action = pol.select_action(ag.Q[state], mask[state])
            nxt, reward, end, _trunc, _info = env.step(action)
            exp = {'state': state, 'action': action, 'reward': reward, 'next_state': nxt, 'terminal': 1 - int(end)}
            mem.store(exp)
            ag.update_q(exp)
            for k, v in zip(('states', 'actions', 'next_states', 'rewards'), (state, action, nxt, reward)):
                got[k].append(v)
            state = nxt
            total += reward
            if end:
                last = nxt
                break
        got['trial_steps'].append(step)
        got['trial_reward'].append(total)
        batch = ag.replay(a['batch'], last)
        idx = [e['action'] * S + e['state'] for e in batch if e['state'] >= 0]
        got['replay'].extend(idx)
        got['replay_len'].append(len(idx))
        mem._T.zero_()                   # self.M.T.fill(0), agent/sfma.py:324
    torch.cuda.synchronize()
    dtypes = {'rewards': np.float64, 'trial_reward': np.float64}
    out = {k: np.array(v, dtype=dtypes.get(k, np.int32)) for k, v in got.items()}
    out.update(Q=ag.Q.cpu().numpy(), Mr=mem.rewards.cpu().numpy(), Ms=mem.states.cpu().numpy(),
               Mt=mem.terminals.cpu().numpy(), C=mem.C.cpu().numpy(), T=mem.T.cpu().numpy(), I=mem.I.cpu().numpy(),
               draws=int(stream.draw_count[0]))
    assert sum(got['replay_len']) > 0
    assert_equal_records(out, golden, KEYS['sfma'], what=name)


@pytest.mark.parametrize('side', [20, 50])
@pytest.mark.parametrize('mode', ['default', 'sweeping'])
def test_memory_replay_with_recency_vs_oracle(side, mode):
    """train(no_replay=True) keeps M.T (20x20: the fused kernel on chip, 50x50: from its workspace); then
    SFMAMemory.replay for a given state and for None, of lengths 1, 12 and 32, and a random batch, must reactivate what
    the oracle does and leave I, the draw counts and Q as it does."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SFMA
    from cobel_rl_b200.memory import SFMAMemory
    from cobel_rl_b200.memory.utils.metrics import Euclidean
    from cobel_rl_b200.misc.gridworld_tools import make_open_field
    from cobel_rl_b200.policy import EpsilonGreedy
    S, n, seed, trials, steps = side * side, 2, 5000 + side, 4, 100
    world = make_open_field(side, side, 0, 1, dense_sas=False)
    W = {'S': S, 'A': 4, 'succ': world['succ'], 'reward': world['rewards'].astype(np.float64),
         'terminal': world['terminals'].astype(np.uint8), 'starts': world['starting_states'].astype(np.int32)}
    metric = Euclidean(side, side)
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    env = Gridworld(world, rng=stream)
    mem = SFMAMemory(metric, S, 4, rng=stream)
    mem.recency, mem.mode = True, mode
    ag = SFMA(env.observation_space, env.action_space, EpsilonGreedy(0.2, rng=stream), mem, rng=stream)
    ag.record = True
    res = ag.train(env, trials, steps, 8, no_replay=True)
    q_before = ag._Q.clone()
    # the state each agent ended in: the most recent experiences (largest T) lie around it
    last_sa = [int(res['step_sa'][i, int(res['n_steps'][i]) - 1]) for i in range(n)]
    given = torch.tensor([int(W['succ'][sa // 4, sa % 4]) for sa in last_sa])
    calls = []
    for length in (1, 12, 32):
        calls.append((length, given, mem.replay(length, given)))
        calls.append((length, None, mem.replay(length, None)))
    rnd = mem.retrieve_random_batch(6, np.ones((S, 4), dtype=bool))
    torch.cuda.synchronize()
    assert torch.equal(ag._Q, q_before), 'the memory-level calls must not touch Q'
    for i in range(n):
        rng = tb.Draws(LazyStream(seed, i), 1)
        st = tb.sfma_init(S, 4)
        tb.sfma_train(W, st, metric.D, rng, trials, steps, 8, policy=('eps', 0.2), no_replay=True, mode=mode,
                      replay_kwargs={'recency': True})
        assert np.array_equal(mem._T[i].cpu().numpy(), st['T']) and float(np.abs(st['T']).sum()) > 0
        total = 0
        for length, state, batch in calls:
            idx = tb.sfma_memory_replay(st, metric.D, rng, length, None if state is None else int(state[i]), mode=mode,
                                        recency=True)
            got = [int(e['action'][i]) * S + int(e['state'][i]) for e in batch if int(e['state'][i]) >= 0]
            assert got == list(idx), 'agent %d, length %d, state %s' % (i, length, state)
            for e, j in zip(batch, idx):
                assert float(e['reward'][i]) == st['Mr'][j % S, j // S]
                assert int(e['next_state'][i]) == st['Ms'][j % S, j // S]
            total += len(idx)
        assert total > 0
        assert np.array_equal(mem._I[i].cpu().numpy(), st['I'])
        assert np.array_equal(mem._C[i].cpu().numpy(), st['C'])
        cdf = np.cumsum(np.ones(S * 4) / (S * 4))
        cdf /= cdf[-1]
        want = [int(cdf.searchsorted(rng.next(), side='right')) for _ in range(6)]
        assert [int(e['action'][i]) * S + int(e['state'][i]) for e in rnd] == want
        assert int(stream.draw_count[i]) == rng.k


def test_agent_replay_with_recency_vs_oracle():
    """SFMA.replay (agent/sfma.py:392-421): the batch from the memory with recency, applied to Q in order."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SFMA
    from cobel_rl_b200.memory import SFMAMemory
    from cobel_rl_b200.memory.utils.metrics import Euclidean
    from cobel_rl_b200.misc.gridworld_tools import make_open_field
    from cobel_rl_b200.policy import EpsilonGreedy
    side, n, seed = 50, 2, 5100
    S = side * side
    world = make_open_field(side, side, 0, 1, dense_sas=False)
    W = {'S': S, 'A': 4, 'succ': world['succ'], 'reward': world['rewards'].astype(np.float64),
         'terminal': world['terminals'].astype(np.uint8), 'starts': world['starting_states'].astype(np.int32)}
    metric = Euclidean(side, side)
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    env = Gridworld(world, rng=stream)
    mem = SFMAMemory(metric, S, 4, rng=stream)
    mem.recency = True
    ag = SFMA(env.observation_space, env.action_space, EpsilonGreedy(0.2, rng=stream), mem, rng=stream)
    ag.train(env, 3, 100, 8, no_replay=True)
    batch = ag.replay(32, None)
    torch.cuda.synchronize()
    for i in range(n):
        rng = tb.Draws(LazyStream(seed, i), 1)
        st = tb.sfma_init(S, 4)
        tb.sfma_train(W, st, metric.D, rng, 3, 100, 8, policy=('eps', 0.2), no_replay=True,
                      replay_kwargs={'recency': True})
        idx = tb.sfma_memory_replay(st, metric.D, rng, 32, None, recency=True)
        assert len(idx) > 0
        for j in idx:
            ea, es = divmod(j, S)
            st['td_acc'] += abs(tb._td_update(st['Q'], es, ea, st['Mr'][es, ea], int(st['Ms'][es, ea]),
                                              int(st['Mt'][es, ea]), 0.99, 0.99, None))
        assert [int(e['action'][i]) * S + int(e['state'][i]) for e in batch if int(e['state'][i]) >= 0] == list(idx)
        assert np.array_equal(ag._Q[i].cpu().numpy(), st['Q'])
        assert float(ag._td[i]) == st['td_acc']
        assert int(stream.draw_count[i]) == rng.k
