"""GPU: the step of dynaq_warp_kernel<A, PLAIN> (csrc/dynaq.cu) reads the replay gather before the action selection
and the step's store; the lane whose replay index is the stored (s,a) takes the stored values.  The result must be the
sequential one bit for bit.  The PLAIN kernel runs on generated streams only, so that lane is made frequent by tiny
worlds (S*A = 16 and 12, and a terminal next to the start, where many trials end on their first step) and many
agents; profiles/step_overlap.py counts the cases on the compared agents, so the test shows that they ran."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import tabular as tb
from oracle.philox import LazyStream

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'profiles'))
import step_overlap  # noqa: E402

pytestmark = pytest.mark.gpu


def worlds():
    from cobel_rl_b200.misc.gridworld_tools import make_gridworld
    return {
        'field2x2': make_gridworld(2, 2, terminals=[0], rewards=np.array([[0, 1]]), goals=[0]),
        'track1x3': make_gridworld(1, 3, terminals=[0], rewards=np.array([[0, 1]]), goals=[0]),
        # the start is next to the terminal: many trials end on their first step
        'goal_next_to_start': make_gridworld(3, 3, terminals=[1], rewards=np.array([[1, 1]]), goals=[1],
                                             starting_states=[0]),
    }


def bits(x):
    return np.asarray(x, dtype=np.float64).view(np.int64)


def run_cuda(world, n, seed, trials, steps):
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import DynaQ
    from cobel_rl_b200.policy import EpsilonGreedy
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    env = Gridworld(world, rng=stream)
    ag = DynaQ(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream))
    res = ag.train(env, trials, steps, 32)            # no trace buffers: the PLAIN kernel
    torch.cuda.synchronize()
    tables = {'Q': ag._Q.cpu().numpy(), 'Mr': ag.M._rewards.cpu().numpy(), 'Ms': ag.M._states.cpu().numpy(),
              'Mt': ag.M._terminals.cpu().numpy()}
    return res, tables, stream.draw_count.cpu().numpy()


# 259 agents: the last CTA of four warps holds three
@pytest.mark.parametrize('name', ['field2x2', 'track1x3', 'goal_next_to_start'])
def test_overlapped_step_matches_the_oracle(name):
    world = worlds()[name]
    W = tb.compile_gridworld(world)
    n, trials = 259, 12
    ids = [0, 1, 2, 3, 97, 128, 255, 256, 257, 258]
    counts = dict.fromkeys(step_overlap.CASES, 0)
    first_step_ends = 0
    for seed in (0x5EED, 7, 1234):
        for steps in (1, 2, 30):
            res, tables, draws = run_cuda(world, n, seed, trials, steps)
            for i in ids:
                st = tb.dynaq_init(W['S'], W['A'])
                rng = tb.Draws(LazyStream(seed, i), 1)
                rec = tb.dynaq_train(W, st, rng, trials, steps, 32).arrays()
                what = '%s seed %d steps %d agent %d' % (name, seed, steps, i)
                assert np.array_equal(res['trial_steps'][i].cpu().numpy(), rec['trial_steps']), what
                assert np.array_equal(bits(res['trial_reward'][i].cpu().numpy()), bits(rec['trial_reward'])), what
                assert int(res['n_steps'][i]) == len(rec['states']), what
                assert int(res['n_replay'][i]) == 32 * len(rec['states']), what
                for key in ('Q', 'Mr'):
                    assert np.array_equal(bits(tables[key][i]), bits(st[key])), '%s: %s' % (what, key)
                assert np.array_equal(tables['Ms'][i], st['Ms']) and np.array_equal(tables['Mt'][i], st['Mt']), what
                assert int(draws[i]) == rng.k, what
                # the kernel's order on the CPU (asserts itself against the sequential order) counts the cases
                step_overlap.run(W, seed, i, trials, steps, counts)
                if steps > 1:
                    first_step_ends += int((rec['trial_steps'] == 0).sum())
    for case in ('gather_fixup', 'trial_end'):
        assert counts[case] > 0, '%s: %s never occurred' % (name, case)
    if name == 'goal_next_to_start':
        assert first_step_ends > 0


@pytest.mark.parametrize('A', [2, 3, 6, 8])
def test_overlapped_step_on_graphs_matches_the_oracle(A):
    """The same loop with the other action counts (A > 4 selects without the tie-pattern table)."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Topology
    from cobel_rl_b200.agent import DynaQ
    from cobel_rl_b200.policy import EpsilonGreedy
    from test_random_worlds_gpu import random_graph
    rs = np.random.default_rng(40 + A)
    nodes, starts = random_graph(rs, 5, A)
    W = tb.compile_topology(nodes, starts)
    n, trials, steps, seed = 67, 10, 25, 900 + A
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    env = Topology(nodes, starts, rng=stream, discrete=True)
    ag = DynaQ(env.observation_space, env.action_space, EpsilonGreedy(0.2, rng=stream))
    res = ag.train(env, trials, steps, 32)
    torch.cuda.synchronize()
    for i in (0, 1, 33, 64, 65, 66):
        st = tb.dynaq_init(W['S'], A)
        rng = tb.Draws(LazyStream(seed, i), 1)
        rec = tb.dynaq_train(W, st, rng, trials, steps, 32, policy=('eps', 0.2)).arrays()
        what = 'A=%d agent %d' % (A, i)
        assert np.array_equal(res['trial_steps'][i].cpu().numpy(), rec['trial_steps']), what
        assert np.array_equal(bits(ag.Q[i].cpu().numpy()), bits(st['Q'])), what
        assert np.array_equal(bits(ag.M.rewards[i].cpu().numpy()), bits(st['Mr'])), what
        assert int(stream.draw_count[i]) == rng.k, what
