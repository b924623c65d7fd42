"""GPU: dynaq_warp_kernel<A, PLAIN, false, SUM> (csrc/dynaq.cu, A <= 4) keeps each state's row maximum V[s] and tie
pattern P[s] on chip and selects actions, builds the online target and runs the replay's speculative pass from them.
Training must give the sequential result bit for bit: Q, M, trial steps and rewards and draw counts against
oracle/tabular.py.  Preset tables with exact ties, -0.0 / +0.0 mixes and negative values test the stage-in and the tie
patterns; profiles/row_summaries.py runs the compared agents on the CPU in the kernel's order (asserting V and P after
every step) and counts the refresh cases, so the test shows that they ran."""
import os
import re
import sys

import numpy as np
import pytest
import torch

from oracle import tabular as tb
from oracle.philox import LazyStream

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'profiles'))
import row_summaries  # noqa: E402

pytestmark = pytest.mark.gpu

MAX_SMEM = 227 * 1024          # kMaxSmem (csrc/common.cuh)


def bits(x):
    return np.asarray(x, dtype=np.float64).view(np.int64)


def preset_q(rs, n, S, A):
    """Values from a small set, so that rows hold exact ties, -0.0 next to +0.0 and negative maxima."""
    vals = np.array([-0.0, 0.0, -1.0, -0.5, 0.25, 1.0])
    return vals[rs.integers(0, len(vals), (n, S, A))]


def train(env_of, n, seed, trials, steps, Q0, profile=False):
    import cobel_rl_b200 as cb
    from cobel_rl_b200.agent import DynaQ
    from cobel_rl_b200.policy import EpsilonGreedy
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    env = env_of(stream)
    ag = DynaQ(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream))
    ag.Q = torch.as_tensor(Q0, device='cuda:0')
    names = []
    if profile:
        from torch.profiler import ProfilerActivity, profile as prof
        with prof(activities=[ProfilerActivity.CUDA]) as p:
            res = ag.train(env, trials, steps, 32)            # no trace buffers: the PLAIN kernels
            torch.cuda.synchronize()
        names = [e.name for e in p.events() if 'dynaq' in e.name]
    else:
        res = ag.train(env, trials, steps, 32)
    torch.cuda.synchronize()
    tables = {'Q': ag._Q.cpu().numpy(), 'Mr': ag.M._rewards.cpu().numpy(), 'Ms': ag.M._states.cpu().numpy(),
              'Mt': ag.M._terminals.cpu().numpy()}
    return res, tables, stream.draw_count.cpu().numpy(), names


def check(W, res, tables, draws, Q0, seed, trials, steps, ids, counts, what):
    for i in ids:
        st = tb.dynaq_init(W['S'], W['A'])
        st['Q'][:] = Q0[i]
        rng = tb.Draws(LazyStream(seed, i), 1)
        rec = tb.dynaq_train(W, st, rng, trials, steps, 32).arrays()
        w = '%s agent %d' % (what, i)
        assert np.array_equal(res['trial_steps'][i].cpu().numpy(), rec['trial_steps']), w
        assert np.array_equal(bits(res['trial_reward'][i].cpu().numpy()), bits(rec['trial_reward'])), w
        assert int(res['n_steps'][i]) == len(rec['states']), w
        for key in ('Q', 'Mr'):
            assert np.array_equal(bits(tables[key][i]), bits(st[key])), '%s: %s' % (w, key)
        assert np.array_equal(tables['Ms'][i], st['Ms']) and np.array_equal(tables['Mt'][i], st['Mt']), w
        assert int(draws[i]) == rng.k, w
        if counts is not None:
            row_summaries.run(W, seed, i, trials, steps, counts, Q0=Q0[i])


def gridworld_env(world):
    from cobel_rl_b200.interface import Gridworld
    return lambda stream: Gridworld(world, rng=stream)


# 259 agents: the last CTA of four warps holds three
@pytest.mark.parametrize('preset', [False, True])
def test_summaries_on_gridworlds_match_the_oracle(preset):
    from cobel_rl_b200.misc.gridworld_tools import make_gridworld
    # walls all round: moves into them are self-loops (s2 == s)
    world = make_gridworld(3, 3, terminals=[8], rewards=np.array([[8, 1], [4, -0.5]]), goals=[8])
    W = tb.compile_gridworld(world)
    n, trials, steps, seed = 259, 20, 25, 0x5EED
    rs = np.random.default_rng(11)
    Q0 = preset_q(rs, n, W['S'], W['A']) if preset else np.zeros((n, W['S'], W['A']))
    res, tables, draws, _ = train(gridworld_env(world), n, seed, trials, steps, Q0)
    counts = dict.fromkeys(row_summaries.CASES, 0)
    check(W, res, tables, draws, Q0, seed, trials, steps, [0, 1, 2, 97, 255, 256, 257, 258], counts,
          'preset %s' % preset)
    for case in ('online_refresh', 'online_self_loop', 'max_changed', 'pattern_changed', 'nonnull_batches',
                 'round_same_state'):
        assert counts[case] > 0, '%s never occurred' % case


@pytest.mark.parametrize('A', [2, 3, 4])
def test_summaries_on_graphs_match_the_oracle(A):
    from cobel_rl_b200.interface import Topology
    from test_random_worlds_gpu import random_graph
    rs = np.random.default_rng(70 + A)
    nodes, starts = random_graph(rs, 6, A)
    W = tb.compile_topology(nodes, starts)
    n, trials, steps, seed = 259, 15, 20, 300 + A
    Q0 = preset_q(rs, n, W['S'], A)
    res, tables, draws, _ = train(lambda stream: Topology(nodes, starts, rng=stream, discrete=True), n, seed, trials,
                                  steps, Q0)
    counts = dict.fromkeys(row_summaries.CASES, 0)
    check(W, res, tables, draws, Q0, seed, trials, steps, [0, 1, 128, 258], counts, 'A=%d' % A)
    assert counts['online_refresh'] > 0 and counts['nonnull_batches'] > 0


def smem_bytes(S, A, K, sums):
    """Dynamic shared memory of a 4-warp CTA of the PLAIN kernel (WorldSmem + 4 x AgentSmem, csrc/dynaq.cu)."""
    SA = S * A
    world = (S * 8 + SA * 4 + K * 4 + S + 15) & ~15
    ptab = (SA * 8 * 2 + S * 8 + SA * 2 + 15) & ~15
    vmax = ptab + 64 * 8 + 256 * 8
    agent = (vmax + S * 8 + S + 15) & ~15 if sums else vmax
    return world + 4 * agent


@pytest.mark.parametrize('side', ['fits', 'above'])
def test_world_at_the_summary_limit(side):
    """The largest gridworld (one row wide) whose CTA fits with the summaries runs the summary kernel; one state more
    runs the PLAIN kernel without them (which still fits), and both stay exact."""
    from cobel_rl_b200.misc.gridworld_tools import make_gridworld
    A = 4
    S = max(x for x in range(2, 2000) if smem_bytes(x, A, x - 1, True) <= MAX_SMEM)
    if side == 'above':
        S += 1
        assert smem_bytes(S, A, S - 1, False) <= MAX_SMEM
    world = make_gridworld(1, S, terminals=[0], rewards=np.array([[0, 1]]), goals=[0])
    W = tb.compile_gridworld(world)
    assert W['S'] == S and len(W['starts']) == S - 1
    n, trials, steps, seed = 9, 3, 40, 77
    Q0 = preset_q(np.random.default_rng(5), n, S, A)
    res, tables, draws, names = train(gridworld_env(world), n, seed, trials, steps, Q0, profile=True)
    args = [re.sub(r'^\((int|bool)\)', '', x.strip()).replace('true', '1').replace('false', '0')
            for x in re.findall(r'dynaq_warp_kernel<([^>]*)>', ' '.join(names))[0].split(',')]
    assert args == ['4', '1', '0', '1' if side == 'fits' else '0'], names
    check(W, res, tables, draws, Q0, seed, trials, steps, [0, 4, 8], None, 'S=%d' % S)
