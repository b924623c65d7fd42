"""GPU: compact SR agent with visited sets beyond shared memory (sr_compact_large_kernel).  A
max_visited above the on-chip limit (900 at 4 actions, 685 at 6) selects the HBM-resident path; it must
compute exactly what the on-chip path and the dense oracle compute."""
import numpy as np
import pytest
import torch

from oracle import cases, tabular as tb
from oracle.philox import LazyStream
from helpers import assert_equal_records, policy_obj, unpack_run

pytestmark = pytest.mark.gpu


def _compact_run(world, n, seed, policy, max_visited, sessions, lr=0.2, gamma=0.95, mask=None, split=None):
    """Runs the (train|test, trials, steps) sessions on one compact SR agent; returns per-session records and
    the final tables."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SR
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    env = Gridworld(world, rng=stream)
    ag = SR(env.observation_space, env.action_space, policy_obj(policy, stream), None, lr, gamma,
            compact=True, max_visited=max_visited)
    ag.record = True
    ag.trials_per_launch = split
    if mask is not None:
        ag.action_mask = mask
    runs = []
    for kind, trials, steps in sessions:
        res = (ag.train if kind == 'train' else ag.test)(env, trials, steps)
        runs.append({k: res[k].cpu().numpy().copy() for k in ('step_sa', 'step_next', 'trial_steps', 'trial_reward',
                                                              'n_steps') if k in res})
    torch.cuda.synchronize()
    return ag, stream, runs


def _tables(ag, i):
    v = int(ag.n_visited[i])
    return {'visited': ag.visited[i, :v].cpu().numpy(), 'SRc': ag.SR_compact[i, :v, :v].cpu().numpy(),
            'rewards': ag.rewards[i, :v].cpu().numpy(), 'model': ag.model[i, :v].cpu().numpy()}


def _open_world(h, w):
    from cobel_rl_b200.misc.gridworld_tools import make_gridworld
    S = h * w
    return make_gridworld(h, w, terminals=[0], rewards=np.array([[0, 1.0], [S // 3, 0.5]]),
                          starting_states=[w + 1, S // 2], dense_sas=False)


@pytest.mark.parametrize('policy,split,masked', [(('eps', 0.3), None, False), (('xeps', 0.3), 2, False),
                                                  (('softmax', 3.0), None, False), (('eps', 0.3), 3, True)])
def test_large_path_equals_on_chip_path(policy, split, masked):
    """Same seeds with max_visited=512 (on chip) and 4096 (HBM path) on 50x50: trajectories, per-trial steps
    and rewards, draw counts and the visited / SRc / rewards / model tables are bit-identical, through
    train() then test(), with and without trials_per_launch and a shared action mask."""
    world = _open_world(50, 50)
    mask = None
    if masked:
        mask = np.ones((2500, 4), dtype=bool)
        mask[::3, 1] = False
        mask[1::5, 2] = False
        mask = torch.as_tensor(mask)
    sessions = [('train', 6, 60), ('test', 2, 40)]
    got = []
    for V in (512, 4096):
        ag, stream, runs = _compact_run(world, 3, 4242, policy, V, sessions, mask=mask, split=split)
        assert int(ag.n_visited.max()) < 512
        got.append((ag, stream.draw_count.cpu().numpy().copy(), runs))
    (a0, d0, r0), (a1, d1, r1) = got
    assert np.array_equal(d0, d1)
    for x, y in zip(r0, r1):
        for k in x:
            assert np.array_equal(x[k], y[k]), k
    for i in range(3):
        t0, t1 = _tables(a0, i), _tables(a1, i)
        for k in t0:
            assert np.array_equal(t0[k], t1[k]), '%s of agent %d' % (k, i)


def _check_vs_oracle(ag, res, i, W, rng, st, trials, steps, policy, A, lr, gamma, learn=True, what=''):
    rec = tb.sr_train(W, st, rng, trials, steps, policy=policy, lr=lr, gamma=gamma, learn=learn).arrays()
    got = unpack_run(res, i, A, W['succ'], W['reward'])
    assert_equal_records(got, rec, ['states', 'actions', 'next_states', 'trial_steps', 'trial_reward'], what=what)
    S = W['S']
    assert np.array_equal(ag.dense_sr(i).cpu().numpy(), st['SR']), 'SR ' + what
    assert np.array_equal(ag.dense_rewards(i).cpu().numpy(), st['rew']), 'rewards ' + what
    v = int(ag.n_visited[i])
    vis = ag.visited[i, :v].cpu().numpy()
    model_dense = np.tile(np.arange(S).reshape(S, 1), A)
    model_dense[vis] = vis[ag.model[i, :v].cpu().numpy()]
    assert np.array_equal(model_dense, st['model']), 'model ' + what


def test_large_path_beyond_on_chip_cap_matches_dense_oracle():
    """60x60 open field with a reward on every fourth state, max_visited=3600: a random walker (eps = 1)
    visits far more than the 900 states that fit on chip; train() then test() are bit-equal to the dense
    oracle (trajectories, draws, SR, rewards, model)."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SR
    from cobel_rl_b200.policy import EpsilonGreedy
    from cobel_rl_b200.misc.gridworld_tools import make_gridworld
    h = w = 60
    S = h * w
    ids = np.arange(S)[::4]
    rw = np.stack([ids, 0.1 + 0.01 * (ids % 17)], axis=1)
    world = make_gridworld(h, w, terminals=[0], rewards=rw, starting_states=[S // 2 + w // 2], dense_sas=False)
    eps = [1.0, 0.3]
    n, trials, steps, lr, gamma = 2, 3, 3000, 0.2, 0.95
    stream = cb.BatchStream(n, seed=31337, device='cuda:0')
    env = Gridworld(world, rng=stream)
    ag = SR(env.observation_space, env.action_space, EpsilonGreedy(eps, rng=stream), None, lr, gamma,
            compact=True, max_visited=S)
    ag.record = True
    res = ag.train(env, trials, steps)
    torch.cuda.synchronize()
    assert int(ag.n_visited.max()) > 900
    W = {'S': S, 'A': 4, 'succ': world['succ'], 'reward': world['rewards'].astype(np.float64),
         'terminal': world['terminals'].astype(np.uint8), 'starts': world['starting_states'].astype(np.int32)}
    states = []
    for i in range(n):
        rng = tb.Draws(LazyStream(31337, i), 1)
        st = tb.sr_init(S, 4)
        _check_vs_oracle(ag, res, i, W, rng, st, trials, steps, ('eps', eps[i]), 4, lr, gamma, what='agent %d' % i)
        assert int(stream.draw_count[i]) == rng.k
        states.append((rng, st))
    rt = ag.test(env, 2, 300)
    torch.cuda.synchronize()
    for i, (rng, st) in enumerate(states):
        _check_vs_oracle(ag, rt, i, W, rng, st, 2, 300, ('eps', eps[i]), 4, lr, gamma, learn=False,
                         what='test() agent %d' % i)
        assert int(stream.draw_count[i]) == rng.k


def test_large_path_stochastic_world_matches_oracle():
    """Slippery 20x20 world (non-deterministic transitions) with max_visited=1000 > 900."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SR
    from cobel_rl_b200.policy import EpsilonGreedy
    from cobel_rl_b200.misc.gridworld_tools import make_gridworld
    world = cases.make_slippery(make_gridworld(20, 20, terminals=[0], rewards=np.array([[0, 1.0], [210, -0.5]]),
                                               starting_states=[21, 230]), 0.25)
    n, trials, steps, lr, gamma = 2, 5, 150, 0.3, 0.9
    stream = cb.BatchStream(n, seed=99, device='cuda:0')
    env = Gridworld(world, rng=stream)
    ag = SR(env.observation_space, env.action_space, EpsilonGreedy(0.4, rng=stream), None, lr, gamma,
            compact=True, max_visited=1000)
    ag.record = True
    res = ag.train(env, trials, steps)
    torch.cuda.synchronize()
    W = tb.compile_gridworld(world)
    for i in range(n):
        rng = tb.Draws(LazyStream(99, i), 1)
        st = tb.sr_init(400, 4)
        _check_vs_oracle(ag, res, i, W, rng, st, trials, steps, ('eps', 0.4), 4, lr, gamma, what='agent %d' % i)
        assert int(stream.draw_count[i]) == rng.k


def test_large_path_six_action_graph_matches_oracle():
    """Hexagonal graph (885 nodes, 6 actions) with max_visited=885 > 685, the on-chip limit at 6 actions."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Topology
    from cobel_rl_b200.agent import SR
    from cobel_rl_b200.policy import EpsilonGreedy
    from cobel_rl_b200.misc.topology_tools import hexagonal
    nodes, starts = hexagonal(30)
    W = tb.compile_topology(nodes, starts)
    S = W['S']
    n, trials, steps, lr, gamma = 2, 4, 300, 0.2, 0.95
    stream = cb.BatchStream(n, seed=6, device='cuda:0')
    env = Topology(nodes, starts, rng=stream, discrete=True)
    ag = SR(env.observation_space, env.action_space, EpsilonGreedy(0.5, rng=stream), None, lr, gamma,
            compact=True, max_visited=S)
    ag.record = True
    res = ag.train(env, trials, steps)
    torch.cuda.synchronize()
    for i in range(n):
        rng = tb.Draws(LazyStream(6, i), 1)
        st = tb.sr_init(S, 6)
        _check_vs_oracle(ag, res, i, W, rng, st, trials, steps, ('eps', 0.5), 6, lr, gamma, what='agent %d' % i)
        assert int(stream.draw_count[i]) == rng.k


def test_large_path_overflow_is_reported():
    """max_visited=1000 on the HBM path: a random walk that leaves the visited set raises CobelError."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200 import _lib
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SR
    from cobel_rl_b200.policy import EpsilonGreedy
    from cobel_rl_b200.misc.gridworld_tools import make_open_field
    stream = cb.BatchStream(2, seed=1, device='cuda:0')
    env = Gridworld(make_open_field(60, 60, 0, 1, dense_sas=False), rng=stream)
    ag = SR(env.observation_space, env.action_space, EpsilonGreedy(1.0, rng=stream), compact=True, max_visited=1000)
    with pytest.raises(_lib.CobelError):
        ag.train(env, 3, 5000)
