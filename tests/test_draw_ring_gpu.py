"""GPU: the PLAIN Dyna-Q and QAgent kernels read their uniforms from a ring of 256 draws in shared memory
(SmemDrawWindowT, csrc/warp_agent.cuh) that a refill extends by the next 192 draws, so no draw is generated twice.
Training must give the sequential result bit for bit: trial steps and rewards, step and replay counts, tables and
the final draw count against oracle/tabular.py.  The cases move the ring's phase: odd and even starting draw counts,
consecutive train() calls that resume mid-ring, one-step trials (a trial start every step, so the parity of the
step's first draw flips each step), runs of many ring wraps, A = 2, 3, 4, and QAgent on the linear track, whose
kernel runs four agents per CTA, with a partial last CTA.  No trace buffers are requested, so the PLAIN kernels run
(for Dyna-Q the row-summary kernel, one agent per CTA)."""
import numpy as np
import pytest
import torch

from oracle import tabular as tb
from oracle.philox import uniforms

pytestmark = pytest.mark.gpu


def bits(x):
    return np.asarray(x, dtype=np.float64).view(np.int64)


class StreamFrom:
    """Draws k0, k0+1, ... of one agent's stream, indexed by stream position (the oracle reads from k0 on)."""

    def __init__(self, seed, agent, k0, n=1 << 17):
        self.k0, self.u = k0, uniforms(seed, agent, n, k0)

    def __getitem__(self, k):
        return self.u[k - self.k0]


def start_counts(n, rs):
    """Starting draw counts of both parities, small and past 2^32 draws (the ring indexes with 32 bits)."""
    k = rs.integers(0, 1000, n)
    k[1::2] |= 1
    k[0::2] &= ~1
    k[3::7] += 1 << 32
    return k


def dynaq_run(env, n, seed, k0, calls):
    import cobel_rl_b200 as cb
    from cobel_rl_b200.agent import DynaQ
    from cobel_rl_b200.policy import EpsilonGreedy
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    e = env(stream)
    ag = DynaQ(e.observation_space, e.action_space, EpsilonGreedy(0.1, rng=stream))
    stream.draw_count.copy_(torch.as_tensor(k0, dtype=torch.int64))     # after the environment's initial reset draw
    out = []
    for trials, steps in calls:
        res = ag.train(e, trials, steps, 32)
        torch.cuda.synchronize()
        out.append({key: v.cpu().numpy() for key, v in res.items() if torch.is_tensor(v)})
    tables = {'Q': ag._Q.cpu().numpy(), 'Mr': ag.M._rewards.cpu().numpy(), 'Ms': ag.M._states.cpu().numpy(),
              'Mt': ag.M._terminals.cpu().numpy()}
    return out, tables, stream.draw_count.cpu().numpy()


def dynaq_check(W, out, tables, draws, seed, k0, calls, ids, what):
    for i in ids:
        st = tb.dynaq_init(W['S'], W['A'])
        rng = tb.Draws(StreamFrom(seed, i, int(k0[i])), int(k0[i]))
        for res, (trials, steps) in zip(out, calls):
            rec = tb.dynaq_train(W, st, rng, trials, steps, 32).arrays()
            w = '%s agent %d' % (what, i)
            assert np.array_equal(res['trial_steps'][i], rec['trial_steps']), w
            assert np.array_equal(bits(res['trial_reward'][i]), bits(rec['trial_reward'])), w
            assert int(res['n_steps'][i]) == len(rec['states']), w
            assert int(res['n_replay'][i]) == 32 * len(rec['states']), w
        for key in ('Q', 'Mr'):
            assert np.array_equal(bits(tables[key][i]), bits(st[key])), '%s agent %d: %s' % (what, i, key)
        assert np.array_equal(tables['Ms'][i], st['Ms']) and np.array_equal(tables['Mt'][i], st['Mt']), what
        assert int(draws[i]) == rng.k, '%s agent %d: draw count' % (what, i)


def open_field():
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.misc.gridworld_tools import make_open_field
    world = make_open_field(5, 5, 0, 1)
    return tb.compile_gridworld(world), lambda stream: Gridworld(world, rng=stream)


@pytest.mark.parametrize('calls', [[(40, 50)], [(7, 50), (1, 3), (12, 50)], [(150, 1)]],
                         ids=['wraps', 'resume', 'one_step'])
def test_dynaq_ring_matches_the_oracle(calls):
    W, env = open_field()
    n, seed = 37, 0xD5A
    k0 = start_counts(n, np.random.default_rng(3))
    out, tables, draws = dynaq_run(env, n, seed, k0, calls)
    # the ring wrapped many times: well over 256 draws per call on average
    assert (draws - k0).min() > 4 * 256
    dynaq_check(W, out, tables, draws, seed, k0, calls, [0, 1, 2, 3, 10, 35, 36], '%s' % calls)


@pytest.mark.parametrize('A', [2, 3, 4])
def test_dynaq_ring_on_graphs(A):
    from cobel_rl_b200.interface import Topology
    from test_random_worlds_gpu import random_graph
    rs = np.random.default_rng(90 + A)
    nodes, starts = random_graph(rs, 6, A)
    W = tb.compile_topology(nodes, starts)
    n, seed, calls = 21, 500 + A, [(9, 20), (6, 20)]
    k0 = start_counts(n, rs)
    out, tables, draws = dynaq_run(lambda stream: Topology(nodes, starts, rng=stream, discrete=True), n, seed, k0,
                                   calls)
    dynaq_check(W, out, tables, draws, seed, k0, calls, [0, 1, 3, 19, 20], 'A=%d' % A)


def test_qagent_ring_on_the_linear_track():
    import cobel_rl_b200 as cb
    from cobel_rl_b200.agent import QAgent
    from cobel_rl_b200.interface import Topology
    from cobel_rl_b200.misc.topology_tools import linear_track
    from cobel_rl_b200.policy import EpsilonGreedy
    nodes, starts = linear_track(10, 2, 1.0, 20.0, 'right')
    W = tb.compile_topology(nodes, starts)
    n, seed, calls = 13, 0x51, [(8, 50), (5, 50)]          # 13 agents: the last CTA of four warps holds one
    k0 = start_counts(n, np.random.default_rng(4))
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    env = Topology(nodes, starts, rng=stream)
    ag = QAgent(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream), rng=stream)
    stream.draw_count.copy_(torch.as_tensor(k0, dtype=torch.int64))     # after the environment's initial reset draw
    out = []
    for trials, steps in calls:
        res = ag.train(env, trials, steps, 32)
        torch.cuda.synchronize()
        out.append({key: v.cpu().numpy() for key, v in res.items() if torch.is_tensor(v)})
    Q, draws = ag.Q.cpu().numpy(), stream.draw_count.cpu().numpy()
    for i in (0, 1, 3, 12):
        st = tb.q_init(W['S'], W['A'])
        rng = tb.Draws(StreamFrom(seed, i, int(k0[i])), int(k0[i]))
        for res, (trials, steps) in zip(out, calls):
            rec = tb.q_train(W, st, rng, trials, steps, 32).arrays()
            w = 'agent %d' % i
            assert np.array_equal(res['trial_steps'][i], rec['trial_steps']), w
            assert np.array_equal(bits(res['trial_reward'][i]), bits(rec['trial_reward'])), w
            assert int(res['n_steps'][i]) == len(rec['states']), w
            assert int(res['n_replay'][i]) == len(rec['replay']), w
        assert np.array_equal(bits(Q[i]), bits(st['Q'])), 'agent %d: Q' % i
        assert int(draws[i]) == rng.k, 'agent %d: draw count' % i
