"""CPU: the oracle restatement against the unmodified reference on seeds / configurations that are not among the
golden cases of oracle/cases.py.  The comparison is with records stored in tests/golden/recorded_records.npz, which
were recorded from the oracle itself after it matched the live reference on these cases (see the provenance note in
tests/helpers.py); with the reference sources present the reference also runs live (oracle/ref_runs.py).  Everything
is bit-equal except PMA's SR = inv(I - gamma T): it comes from LAPACK, whose last bits depend on the host CPU, and is
held to the norm-wise bound of tests/test_pma_gpu.py."""
import numpy as np
import pytest

from cobel_rl_b200.memory.utils.metrics import DR
from oracle import ref_runs, tabular as tb
from oracle.philox import LazyStream
from helpers import KEYS, check_stored_record, make_world

PMA_RTOL = {'SR': 1e-12}


@pytest.mark.parametrize('seed_agent', [(11, 0), (12, 5)])
def test_dynaq_live(seed_agent):
    seed, agent = seed_agent
    world = make_world('walls5')
    ref = lambda: ref_runs.run_dynaq(world, LazyStream(seed, agent), 15, 30, 16, policy=('xeps', 0.3), lr=0.8,
                                     gamma=0.9, mem_lr=0.7)
    W = tb.compile_gridworld(world)
    rng = tb.Draws(LazyStream(seed, agent), 1)
    st = tb.dynaq_init(25, 4)
    got = tb.dynaq_train(W, st, rng, 15, 30, 16, policy=('xeps', 0.3), lr=0.8, gamma=0.9, mem_lr=0.7).arrays()
    got.update(Q=st['Q'], Mr=st['Mr'], Ms=st['Ms'], Mt=st['Mt'], draws=rng.k)
    check_stored_record('dynaq_%d_%d' % seed_agent, got, KEYS['dynaq'], ref)


def test_sr_and_q_live():
    world = make_world('open8')
    W = tb.compile_gridworld(world)
    ref = lambda: ref_runs.run_sr(world, LazyStream(99, 3), 8, 60, policy=('softmax', 4.0), lr=0.4, gamma=0.9)
    rng = tb.Draws(LazyStream(99, 3), 1)
    st = tb.sr_init(64, 4)
    got = tb.sr_train(W, st, rng, 8, 60, policy=('softmax', 4.0), lr=0.4, gamma=0.9).arrays()
    got.update(SR=st['SR'], rew=st['rew'], model=st['model'], draws=rng.k)
    check_stored_record('sr_open8', got, KEYS['sr'], ref)
    ref = lambda: ref_runs.run_q_gridworld(world, LazyStream(99, 3), 8, 40, 12, policy=('eps', 0.25), lr=0.5,
                                           gamma=0.95)
    rng = tb.Draws(LazyStream(99, 3), 1)
    st = tb.q_init(64, 4)
    got = tb.q_train(W, st, rng, 8, 40, 12, policy=('eps', 0.25), lr=0.5, gamma=0.95).arrays()
    got.update(Q=st['Q'], draws=rng.k)
    check_stored_record('q_open8', got, KEYS['q_grid'], ref)


def test_sfma_and_pma_live():
    world = make_world('walls5')
    W = tb.compile_gridworld(world)
    D = DR(5, 5, world['sas'], 0.9, world['invalid_transitions']).D
    ref = lambda: ref_runs.run_sfma(world, D, LazyStream(7, 9), 10, 25, 16, mode='blend_reverse', mask_actions=True,
                                    start_replay=True, nb_replays=2)
    rng = tb.Draws(LazyStream(7, 9), 1)
    st = tb.sfma_init(25, 4)
    got = tb.sfma_train(W, st, D, rng, 10, 25, 16, mode='blend_reverse', mask_actions=True, start_replay=True,
                        nb_replays=2).arrays()
    got.update(Q=st['Q'], Mr=st['Mr'], Ms=st['Ms'], Mt=st['Mt'], C=st['C'], T=st['T'], I=st['I'], draws=rng.k)
    check_stored_record('sfma_blend_reverse', got, KEYS['sfma'], ref)
    # dynamic replay mode (agent/sfma.py:311-318) with two replays per trial
    ref = lambda: ref_runs.run_sfma(world, D, LazyStream(8, 3), 12, 30, 16, mask_actions=True, nb_replays=2,
                                    dynamic=True)
    rng = tb.Draws(LazyStream(8, 3), 1)
    st = tb.sfma_init(25, 4)
    got = tb.sfma_train(W, st, D, rng, 12, 30, 16, mask_actions=True, nb_replays=2, dynamic=True).arrays()
    got.update(Q=st['Q'], Mr=st['Mr'], Ms=st['Ms'], Mt=st['Mt'], C=st['C'], T=st['T'], I=st['I'], draws=rng.k,
               modes=np.array(st['modes'], dtype=np.int32), td=np.float64(st['td_acc']))
    check_stored_record('sfma_dynamic', got, KEYS['sfma'] + ['modes', 'td'], ref)
    ref = lambda: ref_runs.run_pma(world, LazyStream(7, 9), 4, 12, 12, policy=('eps', 0.2), mem_policy=('eps', 0.05),
                                   lr_q=0.7, gamma_q=0.95, mask_actions=True, min_gain_mode='')
    rng = tb.Draws(LazyStream(7, 9), 1)
    st = tb.pma_init(tb.t0_from_succ(W['succ']), 25, 4)
    got = tb.pma_train(W, st, rng, 4, 12, 12, policy=('eps', 0.2), mem_policy=('eps', 0.05), lr_q=0.7, gamma_q=0.95,
                       mask_actions=True, replay_kwargs={'original': False}).arrays()
    got.update(Q=st['Q'], Mr=st['Mr'], Ms=st['Ms'], Mt=st['Mt'], T=st['T'], SR=st['SR'], update_mask=st['update_mask'],
               draws=rng.k)
    check_stored_record('pma_eps', got, KEYS['pma'], ref, rtol=PMA_RTOL)


PMA_SWITCHES = [dict(equal_need=True), dict(equal_gain=True), dict(ignore_barriers=False),
                dict(equal_need=True, equal_gain=True, ignore_barriers=False), dict(allow_loops=True),
                dict(allow_loops=True, equal_need=True)]


@pytest.mark.parametrize('opts', PMA_SWITCHES)
def test_pma_replay_switches_live(opts):
    """PMAMemory.equal_need / equal_gain / ignore_barriers (memory/pma.py:238-249): oracle vs the reference."""
    world = make_world('walls5')
    W = tb.compile_gridworld(world)
    ref = lambda: ref_runs.run_pma(world, LazyStream(11, 2), 3, 15, 10, mask_actions=True, **opts)
    rng = tb.Draws(LazyStream(11, 2), 1)
    st = tb.pma_init(tb.t0_from_succ(W['succ']), 25, 4)
    got = tb.pma_train(W, st, rng, 3, 15, 10, gamma_q=0.99, mask_actions=True, replay_kwargs=dict(opts)).arrays()
    got.update(Q=st['Q'], Mr=st['Mr'], Ms=st['Ms'], Mt=st['Mt'], T=st['T'], SR=st['SR'], update_mask=st['update_mask'],
               draws=rng.k)
    check_stored_record('pma_switches_%d' % PMA_SWITCHES.index(opts), got, KEYS['pma'], ref, rtol=PMA_RTOL)


SFMA_FLAG_CASES = [
    (dict(reward_mod_local=True, reward_modulation=2.5), 'default'),
    (dict(reward_mod=True, reward_modulation=0.5), 'reverse'),
    (dict(state_mod=True), 'default'),
    (dict(C_normalize=True), 'blend_reverse'),
    (dict(D_normalize=True), 'blend_forward'),
    (dict(D_normalize=True, C_normalize=True), 'interpolate'),
    (dict(R_normalize=False, beta=2.0), 'default'),
    (dict(reward_mod_local=True, reward_mod=True, state_mod=True, C_normalize=True, D_normalize=True), 'reverse'),
]


def sfma_flag_kwargs(flags):
    """Reference attribute names -> oracle keyword arguments (store-time flags, replay-time flags)."""
    store = {k: flags[k] for k in ('reward_mod_local', 'reward_mod', 'state_mod', 'reward_modulation') if k in flags}
    names = {'C_normalize': 'c_normalize', 'D_normalize': 'd_normalize', 'R_normalize': 'r_normalize', 'beta': 'beta'}
    return store, {names[k]: flags[k] for k in names if k in flags}


@pytest.mark.parametrize('flags,mode', SFMA_FLAG_CASES)
def test_sfma_modulation_flags_live(flags, mode):
    """SFMAMemory strength modulation and normalisation switches (memory/sfma.py:216-236, 283-288, 319-320)."""
    world = make_world('walls5')
    W = tb.compile_gridworld(world)
    D = DR(5, 5, world['sas'], 0.9, world['invalid_transitions']).D
    ref = lambda: ref_runs.run_sfma(world, D, LazyStream(21, 4), 8, 30, 16, mode=mode, mask_actions=True,
                                    mem_flags=flags)
    rng = tb.Draws(LazyStream(21, 4), 1)
    st = tb.sfma_init(25, 4)
    store, rk = sfma_flag_kwargs(flags)
    got = tb.sfma_train(W, st, D, rng, 8, 30, 16, mode=mode, mask_actions=True, replay_kwargs=rk, **store).arrays()
    got.update(Q=st['Q'], Mr=st['Mr'], Ms=st['Ms'], Mt=st['Mt'], C=st['C'], T=st['T'], I=st['I'], draws=rng.k)
    check_stored_record('sfma_flags_%d' % SFMA_FLAG_CASES.index((flags, mode)), got, KEYS['sfma'], ref)


@pytest.mark.parametrize('k', range(6))
def test_dynaq_random_configurations_live(k):
    """Randomised Dyna-Q configurations (policy kind and parameter, masks, replay schedule, batch, learning rates)
    on the maze templates: the oracle against the unmodified reference."""
    from cobel_rl_b200.misc import gridworld_tools as tools
    rs = np.random.default_rng(300 + k)
    world = [tools.make_t_maze(3, 2), tools.make_double_t_maze(2, 1), tools.make_8_maze(3, 2),
             tools.make_cross_maze(2, 2, 'left'), tools.make_detour_maze(1, 1, 2, 2),
             tools.make_two_choice_t_maze(3, 3, 1)][k]
    S = world['states']
    kind = ['eps', 'xeps', 'softmax'][k % 3]
    par = float(np.round(rs.uniform(0.05, 0.5) if kind != 'softmax' else rs.uniform(0.5, 3.0), 3))
    kw = dict(policy=(kind, par), lr=float(np.round(rs.uniform(0.3, 1.0), 3)), gamma=float(np.round(rs.uniform(0.5, 0.99), 3)),
              mem_lr=float(np.round(rs.uniform(0.3, 1.0), 3)), mask_actions=bool(k % 2),
              no_replay=(k == 4), episodic_replay=(k == 5))
    batch = int(rs.choice([4, 16, 32]))
    W = tb.compile_gridworld(world)
    mask = tb.valid_move_mask(W['succ'])
    mask[np.arange(S), 0] |= ~mask.any(axis=1)        # dead-end cells keep one valid action
    ref = lambda: ref_runs.run_dynaq(world, LazyStream(40 + k, 1), 10, 25, batch,
                                     action_mask=mask if kw['mask_actions'] else None, **kw)
    rng = tb.Draws(LazyStream(40 + k, 1), 1)
    st = tb.dynaq_init(S, 4)
    st['action_mask'] = mask
    got = tb.dynaq_train(W, st, rng, 10, 25, batch, **kw).arrays()
    got.update(Q=st['Q'], Mr=st['Mr'], Ms=st['Ms'], Mt=st['Mt'], draws=rng.k)
    check_stored_record('dynaq_random_%d' % k, got, KEYS['dynaq'], ref)
