"""GPU: the stand-alone methods of the compact SR agent (cobel_sr_compact_op, sr_compact_op_kernel).

``SR(..., compact=True).update / retrieve_q / predict_on_batch`` must compute what the dense agent computes: a
hand-written loop lands on the dense goldens, stand-alone steps interleave with fused ``train()`` without a trace,
and Q of every state (visited or not) equals the dense agent's, on the on-chip and the HBM-resident path alike."""
import numpy as np
import pytest
import torch

from oracle import cases, tabular as tb
from helpers import TRAJ, assert_equal_records, load_golden, make_world, policy_obj, unpack_run

pytestmark = pytest.mark.gpu


def _model_dense(ag, i, S, A):
    """The dense [S, A] successor model implied by the compact tables of agent i."""
    v = int(ag._n_visited[i])
    vis = ag._visited[i, :v].cpu().numpy()
    out = np.tile(np.arange(S, dtype=np.int32).reshape(S, 1), A)
    out[vis] = vis[ag._model[i, :v].cpu().numpy()]
    return out


def _tables(ag, i):
    v = int(ag._n_visited[i])
    return {'n_visited': v, 'visited': ag._visited[i, :v].cpu().numpy(), 'SRc': ag._SRc[i, :v, :v].cpu().numpy(),
            'rewards': ag._rewards[i, :v].cpu().numpy(), 'model': ag._model[i, :v].cpu().numpy()}


def _hand_written_trials(env, pol, ag, trials, steps, mask=None):
    """The reference's SR loop (agent/sr.py:166-190) driven through the stand-alone methods; returns the trajectory."""
    s_, a_, s2_, r_, tsteps, trew = [], [], [], [], [], []
    for _ in range(trials):
        state, _info = env.reset()
        total, step = 0.0, 0
        for step in range(steps):
            action = pol.select_action(ag.retrieve_q(state), mask[state] if mask is not None else None)
            nxt, reward, end, _trunc, _info = env.step(action)
            ag.update({'state': state, 'action': action, 'reward': reward, 'next_state': nxt, 'terminal': 1 - int(end)})
            s_.append(state); a_.append(action); s2_.append(nxt); r_.append(reward)
            state = nxt
            total += reward
            if end:
                break
        tsteps.append(step); trew.append(total)
    return {'states': np.array(s_, dtype=np.int32), 'actions': np.array(a_, dtype=np.int32),
            'next_states': np.array(s2_, dtype=np.int32), 'rewards': np.array(r_, dtype=np.float64),
            'trial_steps': np.array(tsteps, dtype=np.int32), 'trial_reward': np.array(trew, dtype=np.float64)}


@pytest.mark.parametrize('max_visited', ['S', 2048])
@pytest.mark.parametrize('name', ['sr_open5', 'sr_walls5_mask', 'sr_slip5', 'sr_open13'])
def test_compact_hand_written_loop_matches_golden(name, max_visited):
    """tests/test_standalone_gpu.py's dense hand-written SR loop with a compact agent: trajectories, draws and the
    implied dense SR / rewards / model equal the golden bit for bit.  max_visited = 2048 changes the row stride of SRc
    and lies above the on-chip cap of the fused kernel."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SR
    _kind, wname, case_agent, args = cases.CASES[name]
    a = dict(args)
    stream = cb.BatchStream(None, seed=cases.SEED, device='cuda:0', agent_id_base=case_agent)
    env = Gridworld(make_world(wname), rng=stream)
    S = env.n_states
    pol = policy_obj(a.get('policy', ('eps', 0.1)), stream)
    ag = SR(env.observation_space, env.action_space, pol, None, a.get('lr', 0.1), a.get('gamma', 0.99), compact=True,
            max_visited=S if max_visited == 'S' else max_visited)
    mask = None
    if a.get('mask_actions'):
        mask = torch.as_tensor(tb.valid_move_mask(env._succ.cpu().numpy()), device='cuda:0')
    got = _hand_written_trials(env, pol, ag, a['trials'], a['steps'], mask)
    torch.cuda.synchronize()
    got.update(SR=ag.dense_sr(0).cpu().numpy(), rew=ag.dense_rewards(0).cpu().numpy(), model=_model_dense(ag, 0, S, 4),
               draws=int(stream.draw_count[0]))
    assert_equal_records(got, load_golden(name), TRAJ + ['SR', 'rew', 'model', 'draws'], what=name)


def _open_world(h, w):
    from cobel_rl_b200.misc.gridworld_tools import make_gridworld
    S = h * w
    return make_gridworld(h, w, terminals=[0], rewards=np.array([[0, 1.0], [S // 3, 0.5]]),
                          starting_states=[w + 1, S // 2], dense_sas=False)


@pytest.mark.parametrize('max_visited', [512, 4096])
@pytest.mark.parametrize('policy', [('eps', 0.3), ('softmax', 3.0)], ids=['eps', 'softmax'])
def test_stand_alone_steps_interleave_with_fused_training(policy, max_visited):
    """50x50, single-agent streams of several agent ids.  Agent A trains 3 trials fused, 2 by hand, 3 fused again;
    agent B (same id) trains all 8 fused.  Visited order, n_visited, SRc, rewards, model, trajectories and draw counts
    are bit-identical, with the fused parts on the on-chip kernel (512) and on the HBM kernel (4096)."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SR
    world = _open_world(50, 50)
    k, m, rest, steps = 3, 2, 3, 60

    def agent(agent_id):
        stream = cb.BatchStream(None, seed=2024, device='cuda:0', agent_id_base=agent_id)
        env = Gridworld(world, rng=stream)
        pol = policy_obj(policy, stream)
        ag = SR(env.observation_space, env.action_space, pol, None, 0.2, 0.95, compact=True, max_visited=max_visited)
        ag.record = True
        return stream, env, pol, ag

    def fused(ag, env, trials):
        res = ag.train(env, trials, steps)
        rec = unpack_run(res, 0, 4, world['succ'], world['rewards'].astype(np.float64))
        return {key: rec[key] for key in TRAJ}

    for agent_id in (0, 7, 93):
        sa, ea, pa, A = agent(agent_id)
        parts = [fused(A, ea, k), _hand_written_trials(ea, pa, A, m, steps), fused(A, ea, rest)]
        got = {key: np.concatenate([p[key] for p in parts]) for key in TRAJ}
        sb, eb, _pb, B = agent(agent_id)
        want = fused(B, eb, k + m + rest)
        torch.cuda.synchronize()
        what = 'agent %d, %s, max_visited %d' % (agent_id, policy[0], max_visited)
        assert int(A._n_visited[0]) < 512, what
        assert_equal_records(got, want, TRAJ, what=what)
        assert int(sa.draw_count[0]) == int(sb.draw_count[0]), what
        ta, tb_ = _tables(A, 0), _tables(B, 0)
        for key in ta:
            assert np.array_equal(ta[key], tb_[key]), '%s: %s' % (what, key)


def _q_worlds():
    from cobel_rl_b200.misc.gridworld_tools import make_gridworld
    ids = np.arange(1600)[::4]
    many = np.stack([ids, np.where(ids % 3 == 0, -1.0, 1.0) * (0.1 + 0.01 * (ids % 17))], axis=1)
    return {
        '20x20': make_gridworld(20, 20, terminals=[0], rewards=np.array([[0, 1.0], [210, 0.5]]),
                                starting_states=[21, 230], dense_sas=False),
        'negative': make_gridworld(20, 20, terminals=[0], rewards=np.array([[0, 1.0], [57, -0.5], [133, -1.0],
                                                                            [300, -0.25]]),
                                   starting_states=[21, 230], dense_sas=False),
        '40x40_many': make_gridworld(40, 40, terminals=[0], rewards=many, starting_states=[820], dense_sas=False),
    }


def _trained_pair(make_env, S, n, seed, trials, steps, max_visited):
    """A dense and a compact SR agent trained on streams with the same seed (identical runs)."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.agent import SR
    from cobel_rl_b200.policy import EpsilonGreedy
    out = []
    for compact in (False, True):
        stream = cb.BatchStream(n, seed=seed, device='cuda:0')
        env = make_env(stream)
        pol = EpsilonGreedy(np.linspace(0.1, 0.6, n).tolist(), rng=stream)
        ag = SR(env.observation_space, env.action_space, pol, None, 0.2, 0.95, compact=compact, max_visited=max_visited)
        ag.train(env, trials, steps)
        out.append((stream, ag))
    torch.cuda.synchronize()
    return out


def _check_q_against_dense(dense, compact, S, A, seed):
    want = dense.predict_on_batch(range(S))
    got = compact.predict_on_batch(range(S))
    assert got.shape == (dense._stream.n_agents, S, A)
    assert np.array_equal(got.cpu().numpy(), want.cpu().numpy())
    n = compact._stream.n_agents
    states = torch.as_tensor(np.random.default_rng(seed).integers(0, S, n), device='cuda:0')
    q = compact.retrieve_q(states).cpu().numpy()
    assert q.shape == (n, A)
    for i in range(n):
        st = {'SR': dense.SR[i].cpu().numpy(), 'rew': dense.rewards[i].cpu().numpy(),
              'model': dense.model[i].cpu().numpy()}
        assert np.array_equal(q[i], tb.sr_retrieve_q(st, int(states[i]))), 'agent %d' % i


@pytest.mark.parametrize('world', ['20x20', 'negative', '40x40_many'])
def test_predict_on_batch_equals_dense_agent(world):
    """64 agents, dense and compact trained on the same stream: predict_on_batch(range(S)) is equal, including the
    states an agent never visited; retrieve_q with one state per agent equals the oracle on the dense tables.
    The 40x40 world carries rewards of both signs on 400 states and runs on the HBM path (max_visited = 1600)."""
    from cobel_rl_b200.interface import Gridworld
    w = _q_worlds()[world]
    S = int(np.asarray(w['rewards']).size)
    (_sd, dense), (_sc, compact) = _trained_pair(lambda st: Gridworld(w, rng=st), S, 64, 515, 4, 150, S)
    for i in range(64):
        assert np.array_equal(compact.dense_sr(i).cpu().numpy(), dense.SR[i].cpu().numpy())
    assert int(compact.n_visited.min()) < S
    assert int((compact.rewards != 0).sum(dim=1).max()) > 1
    _check_q_against_dense(dense, compact, S, 4, 1)


def test_predict_on_batch_equals_dense_agent_on_six_action_graph():
    """The 885-node hexagonal graph (6 actions) at max_visited = 885, above the on-chip cap at 6 actions."""
    from cobel_rl_b200.interface import Topology
    from cobel_rl_b200.misc.topology_tools import hexagonal
    nodes, starts = hexagonal(30)
    S = tb.compile_topology(nodes, starts)['S']
    (_sd, dense), (_sc, compact) = _trained_pair(lambda st: Topology(nodes, starts, rng=st, discrete=True), S, 64, 6,
                                                 3, 200, S)
    assert int(compact.n_visited.min()) < S
    _check_q_against_dense(dense, compact, S, 6, 2)


@pytest.mark.parametrize('max_visited', [256, 2048])
def test_calls_leave_state_alone(max_visited):
    """retrieve_q and predict_on_batch change no table and consume no draws; update consumes no draws."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SR
    from cobel_rl_b200.policy import EpsilonGreedy
    stream = cb.BatchStream(8, seed=11, device='cuda:0')
    env = Gridworld(_open_world(30, 30), rng=stream)
    ag = SR(env.observation_space, env.action_space, EpsilonGreedy(0.3, rng=stream), None, 0.2, 0.95, compact=True,
            max_visited=max_visited)
    ag.train(env, 3, 60)
    names = ('_SRc', '_rewards', '_model', '_visited', '_n_visited')
    before = {k: getattr(ag, k).clone() for k in names}
    draws = stream.draw_count.clone()
    ag.retrieve_q(torch.arange(8, device='cuda:0') * 97)
    ag.retrieve_q(31)
    ag.predict_on_batch(range(900))
    torch.cuda.synchronize()
    for k in names:
        assert torch.equal(getattr(ag, k), before[k]), k
    assert torch.equal(stream.draw_count, draws)
    ag.update({'state': 31, 'action': 2, 'reward': 0.5, 'next_state': 899, 'terminal': 1})
    torch.cuda.synchronize()
    assert torch.equal(stream.draw_count, draws)
    assert not torch.equal(ag._n_visited, before['_n_visited'])


def test_q_monitor_on_compact_agent():
    """monitor.QMonitor calls predict_on_batch at the end of every trial: a compact agent's trace equals the dense
    agent's on the same stream."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SR
    from cobel_rl_b200.monitor import QMonitor
    from cobel_rl_b200.policy import EpsilonGreedy
    world = _q_worlds()['20x20']
    traces = []
    for compact in (False, True):
        stream = cb.BatchStream(8, seed=5, device='cuda:0')
        env = Gridworld(world, rng=stream)
        mon = QMonitor(6, [0, 1, 21, 210, 230, 399])
        ag = SR(env.observation_space, env.action_space, EpsilonGreedy(0.2, rng=stream), None, 0.2, 0.95,
                custom_callbacks={'on_trial_end': [mon.update]}, compact=compact, max_visited=400)
        ag.trials_per_launch = 1
        ag.train(env, 6, 80)
        traces.append(mon.get_trace())
    assert len(traces[1]) == 6
    for d, c in zip(*traces):
        assert c.shape == (8, 6, 4) and np.array_equal(d, c)
    assert any(np.any(c != 0) for c in traces[1])


def test_update_beyond_max_visited_raises_the_train_message():
    import cobel_rl_b200 as cb
    from cobel_rl_b200 import _lib
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SR
    from cobel_rl_b200.policy import EpsilonGreedy
    from cobel_rl_b200.misc.gridworld_tools import make_open_field
    stream = cb.BatchStream(2, seed=1, device='cuda:0')
    env = Gridworld(make_open_field(30, 30, 0, 1, dense_sas=False), rng=stream)
    fused = SR(env.observation_space, env.action_space, EpsilonGreedy(1.0, rng=stream), compact=True, max_visited=8)
    with pytest.raises(_lib.CobelError) as train_err:
        fused.train(env, 3, 200)
    ag = SR(env.observation_space, env.action_space, EpsilonGreedy(1.0, rng=stream), compact=True, max_visited=8)
    for s in range(0, 8, 2):
        ag.update({'state': s, 'action': 0, 'reward': 0.0, 'next_state': s + 1, 'terminal': 1})
    assert int(ag.n_visited.min()) == 8
    with pytest.raises(_lib.CobelError) as update_err:
        ag.update({'state': 7, 'action': 1, 'reward': 0.0, 'next_state': 8, 'terminal': 1})
    assert str(update_err.value) == str(train_err.value)
    with pytest.raises(IndexError):
        ag.update({'state': 900, 'action': 1, 'reward': 0.0, 'next_state': 8, 'terminal': 1})
    with pytest.raises(IndexError):
        ag.retrieve_q(-1)


def test_predict_on_batch_of_10000_states_is_one_launch():
    import cobel_rl_b200 as cb
    from cobel_rl_b200 import _lib
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SR
    from cobel_rl_b200.policy import EpsilonGreedy
    from cobel_rl_b200.misc.gridworld_tools import make_open_field
    stream = cb.BatchStream(4, seed=3, device='cuda:0')
    env = Gridworld(make_open_field(100, 100, 0, 1, dense_sas=False), rng=stream)
    ag = SR(env.observation_space, env.action_space, EpsilonGreedy(0.3, rng=stream), compact=True, max_visited=2048)
    ag.train(env, 2, 300)
    L = _lib.lib()
    c0 = L.cobel_launch_count()
    q = ag.predict_on_batch(range(10000))
    assert L.cobel_launch_count() - c0 == 1
    assert q.shape == (4, 10000, 4)
    c0 = L.cobel_launch_count()
    ag.retrieve_q(torch.tensor([5, 17, 1000, 9999]))
    ag.update({'state': 5, 'action': 1, 'reward': 0.0, 'next_state': 6, 'terminal': 1})
    assert L.cobel_launch_count() - c0 == 2
