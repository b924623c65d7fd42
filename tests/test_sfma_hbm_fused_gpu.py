"""GPU: SFMA options that need the fused kernel (recency, decay_strength != 1, reward_mod, train(no_replay=True), test()
of such a memory) on state spaces whose per-agent tables exceed shared memory: sfma_kernel<A, MODS, true> runs on the
same SfmaSmem layout in a global workspace.  Trajectories, replays, tables, |TD| accumulators and draw counts must be
bit-equal to the oracle (oracle/tabular.py: sfma_train), agent by agent with per-agent hyper-parameters."""
import numpy as np
import pytest
import torch

from oracle import tabular as tb
from oracle.philox import LazyStream
from helpers import assert_equal_records, unpack_run

pytestmark = pytest.mark.gpu

LR, GAMMA, MEM_LR, EPS = [0.9, 0.5, 0.99], [0.99, 0.9, 0.95], [0.9, 0.6, 1.0], [0.1, 0.3, 0.05]
# SFMAMemory attributes -> keyword of tb.sfma_train (store side) or of its replay_kwargs (replay side)
STORE = {'decay_strength': 'decay_strength', 'reward_mod_local': 'reward_mod_local', 'reward_mod': 'reward_mod',
         'state_mod': 'state_mod', 'reward_modulation': 'reward_modulation'}
REPLAY = {'recency': 'recency', 'C_normalize': 'c_normalize', 'D_normalize': 'd_normalize', 'R_normalize': 'r_normalize',
          'beta': 'beta'}
AGENT = {'nb_replays': 'nb_replays', 'start_replay': 'start_replay', 'random': 'random_replay', 'dynamic': 'dynamic'}


def _world(side):
    """side x side open field, goal 0, with small rewards on a sparse lattice so that reward modulation acts."""
    from cobel_rl_b200.misc.gridworld_tools import make_open_field
    world = make_open_field(side, side, 0, 1, dense_sas=False)
    world['rewards'] = world['rewards'].astype(np.float64)
    world['rewards'][5::37] = -0.25
    world['rewards'][11::53] = 0.5
    W = {'S': side * side, 'A': 4, 'succ': world['succ'], 'reward': world['rewards'],
         'terminal': world['terminals'].astype(np.uint8), 'starts': world['starting_states'].astype(np.int32)}
    return world, W


def _build(side, n, seed, mem_opts, ag_opts, mask):
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import SFMA
    from cobel_rl_b200.memory import SFMAMemory
    from cobel_rl_b200.memory.utils.metrics import Euclidean
    from cobel_rl_b200.policy import EpsilonGreedy
    world, W = _world(side)
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    env = Gridworld(world, rng=stream)
    mem = SFMAMemory(Euclidean(side, side), side * side, 4, learning_rate=MEM_LR[:n], rng=stream)
    for k, v in mem_opts.items():
        assert hasattr(mem, k), k
        setattr(mem, k, v)
    ag = SFMA(env.observation_space, env.action_space, EpsilonGreedy(EPS[:n], rng=stream), mem, None, LR[:n], GAMMA[:n],
              rng=stream)
    for k, v in ag_opts.items():
        assert hasattr(ag, k), k
        setattr(ag, k, v)
    if mask:
        ag.mask_actions = True
        ag.action_mask = tb.valid_move_mask(W['succ'])
    ag.record = True
    return env, ag, mem, stream, W


def _oracle(W, D, seed, i, trials, steps, batch, mem_opts, ag_opts, mask, no_replay=False, st=None, rng=None):
    rng = rng if rng is not None else tb.Draws(LazyStream(seed, i), 1)
    if st is None:
        st = tb.sfma_init(W['S'], 4)
        if mask:
            st['action_mask'] = tb.valid_move_mask(W['succ'])
    kw = {STORE[k]: v for k, v in mem_opts.items() if k in STORE}
    kw.update({AGENT[k]: v for k, v in ag_opts.items() if k in AGENT})
    rk = {REPLAY[k]: v for k, v in mem_opts.items() if k in REPLAY}
    rec = tb.sfma_train(W, st, D, rng, trials, steps, batch, policy=('eps', EPS[i]), lr=LR[i], gamma=GAMMA[i],
                        mem_lr=MEM_LR[i], mask_actions=mask, mode=mem_opts.get('mode', 'default'), no_replay=no_replay,
                        replay_kwargs=rk, **kw).arrays()
    return rec, st, rng


def _compare(res, ag, mem, stream, W, i, rec, st, rng, what, dynamic=False):
    got = unpack_run(res, i, 4, W['succ'], W['reward'])
    got.update(Q=ag._Q[i].cpu().numpy(), C=mem._C[i].cpu().numpy(), T=mem._T[i].cpu().numpy(),
               I=mem._I[i].cpu().numpy(), td=float(ag._td[i]), draws=int(stream.draw_count[i]))
    rec.update(Q=st['Q'], C=st['C'], T=st['T'], I=st['I'], td=st['td_acc'], draws=rng.k)
    keys = ['states', 'actions', 'trial_steps', 'replay', 'replay_len', 'Q', 'C', 'T', 'I', 'td', 'draws']
    if dynamic:
        # the oracle records the index into ['reverse', 'default']; the kernel reports COBEL_SFMA_* ids (2 = reverse)
        got['modes'] = np.where(res['replay_mode'][i].cpu().numpy() == 2, 0, 1).astype(np.int32)
        rec['modes'] = np.array(st['modes'], dtype=np.int32)
        keys.append('modes')
    assert_equal_records(got, rec, keys, what='%s agent %d' % (what, i))


def _check(side, n, trials, steps, batch, seed, mem_opts, ag_opts=None, mask=False, no_replay=False, what=''):
    ag_opts = ag_opts or {}
    env, ag, mem, stream, W = _build(side, n, seed, mem_opts, ag_opts, mask)
    res = ag.train(env, trials, steps, batch, no_replay=no_replay)
    torch.cuda.synchronize()
    assert int(res['flags'].abs().sum()) == 0, 'flags %s' % res['flags'].tolist()
    assert mem._workspace is not None, 'the tables of this configuration exceed shared memory'
    assert int(res['n_replay'].sum()) > 0 or no_replay
    for i in range(n):
        rec, st, rng = _oracle(W, mem.metric.D, seed, i, trials, steps, batch, mem_opts, ag_opts, mask, no_replay)
        _compare(res, ag, mem, stream, W, i, rec, st, rng, what or str(mem_opts), dynamic=bool(ag_opts.get('dynamic')))
    return ag, mem


@pytest.mark.parametrize('mode', ['default', 'reverse', 'sweeping'])
def test_recency_50x50(mode):
    _check(50, 3, 4, 80, 32, 4001, dict(recency=True, mode=mode))


def test_decay_strength_50x50():
    _check(50, 3, 4, 80, 32, 4002, dict(decay_strength=0.95))


def test_reward_mod_with_the_other_switches_50x50():
    _check(50, 3, 4, 80, 24, 4003, dict(reward_mod=True, reward_mod_local=True, state_mod=True, reward_modulation=0.5,
                                        C_normalize=True, D_normalize=True, R_normalize=False, beta=2.0, mode='reverse'))


def test_no_replay_keeps_T_50x50():
    ag, mem = _check(50, 2, 3, 60, 16, 4004, {}, no_replay=True)
    assert float(mem._T.abs().sum()) > 0


def test_random_replay_with_recency_and_mask_50x50():
    _check(50, 3, 4, 60, 32, 4005, dict(recency=True), dict(random=True), mask=True)


def test_dynamic_start_replay_two_replays_and_mask_50x50():
    _check(50, 3, 4, 80, 24, 4006, dict(decay_strength=0.97, recency=True),
           dict(dynamic=True, start_replay=True, nb_replays=2), mask=True)


def test_test_of_a_memory_with_recency_and_decay_50x50():
    """test() passes no_replay = 1, so the layout includes T: the fused kernel runs from the workspace and learns
    nothing."""
    mem_opts = dict(recency=True, decay_strength=0.95)
    env, ag, mem, stream, W = _build(50, 3, 4007, mem_opts, {}, False)
    ag.train(env, 2, 60, 16)
    tables = [t.clone() for t in (ag._Q, mem._C, mem._T, mem._I, mem._rewards, mem._states, mem._terminals)]
    ws = mem._workspace
    rt = ag.test(env, 3, 60)
    torch.cuda.synchronize()
    assert mem._workspace is ws, 'the workspace is kept across calls'
    assert int(rt['flags'].abs().sum()) == 0
    for a, b in zip(tables, (ag._Q, mem._C, mem._T, mem._I, mem._rewards, mem._states, mem._terminals)):
        assert torch.equal(a, b), 'test() must not change the tables'
    for i in range(3):
        _rec, st, rng = _oracle(W, mem.metric.D, 4007, i, 2, 60, 16, mem_opts, {}, False)
        want = tb.tabular_test(W, st['Q'], rng, 3, 60, policy=('eps', EPS[i])).arrays()
        got = unpack_run(rt, i, 4, W['succ'], W['reward'])
        assert_equal_records(got, want, ['states', 'actions', 'trial_steps'], what='test agent %d' % i)
        assert int(stream.draw_count[i]) == rng.k


def test_trials_per_launch_equals_one_launch_50x50():
    mem_opts = dict(recency=True, decay_strength=0.95)
    runs = []
    for per_launch in (None, 2):
        env, ag, mem, stream, W = _build(50, 2, 4008, mem_opts, {}, False)
        ag.trials_per_launch = per_launch
        res = ag.train(env, 5, 60, 16)
        torch.cuda.synchronize()
        runs.append([unpack_run(res, i, 4, W['succ'], W['reward']) for i in range(2)] +
                    [t.cpu().numpy() for t in (ag._Q, mem._C, mem._T, mem._I, stream.draw_count)])
    for i in range(2):
        assert_equal_records(runs[1][i], runs[0][i], ['states', 'actions', 'trial_steps', 'replay', 'replay_len'],
                             what='agent %d' % i)
    for a, b in zip(runs[0][2:], runs[1][2:]):
        assert np.array_equal(a, b)


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if 'sfma' in e.name}


@pytest.mark.parametrize('side, mem_opts, hbm', [
    (34, dict(recency=True), False), (35, dict(recency=True), True),
    (37, dict(decay_strength=0.95), False), (38, dict(decay_strength=0.95), True)])
def test_boundary_worlds(side, mem_opts, hbm):
    """1191 states with recency, 1428 with decay only (4 actions, 256 threads, batch 32): the largest world on each side
    of the boundary runs the on-chip fused kernel, the next one the HBM instantiation; both match the oracle."""
    env, ag, mem, stream, W = _build(side, 2, 4100 + side, mem_opts, {}, False)
    names = _kernel_names(lambda: ag.train(env, 3, 60, 32))
    res = ag.last_run
    assert int(res['flags'].abs().sum()) == 0
    fused = [n for n in names if 'sfma_kernel<' in n]
    assert fused and all(('sfma_kernel<4, false, %s>' % ('true' if hbm else 'false')) in n for n in fused), names
    assert (mem._workspace is not None) == hbm
    for i in range(2):
        rec, st, rng = _oracle(W, mem.metric.D, 4100 + side, i, 3, 60, 32, mem_opts, {}, False)
        _compare(res, ag, mem, stream, W, i, rec, st, rng, '%dx%d %s' % (side, side, mem_opts))
