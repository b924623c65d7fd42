"""GPU: the Dyna-Q replay drops the updates that provably leave Q bit-identical (td_batch_level_parallel in
csrc/warp_agent.cuh).  Replay batches are placed deliberately through a user stream on preset tables -- all-null
batches, null-looking updates whose inputs an earlier update changes, chains of such updates, write-after-read
pairs, duplicate entries, -0.0 entries and negative rewards -- and compared bit for bit with the sequential
oracle; the two-agents-per-warp kernel is checked on a run of 16385 agents (its last warp half empty)."""
import numpy as np
import pytest
import torch

from oracle import tabular as tb
from oracle.philox import LazyStream
from helpers import make_world, unpack_run

pytestmark = pytest.mark.gpu

S, A = 25, 4
LR, GAMMA = 0.99, 0.99
START = 12                          # every case starts here; its first step moves to state 11 (action 0)
FILLER = [(24, 0), (24, 1), (24, 2), (24, 3), (19, 0), (19, 1), (19, 2), (19, 3)]     # null on the base tables


def world():
    return make_world('open5')


def bits(x):
    return np.asarray(x, dtype=np.float64).view(np.int64)


def case_all_null(st):
    Q, Mr, Ms, Mt = st['Q'], st['Mr'], st['Ms'], st['Mt']
    Q[5, 1] = Mr[5, 1] = 0.75                                     # at its fixed point (terminal transition)
    Ms[8, 0], Mt[8, 0], Q[8, 0] = 5, 1, GAMMA * 1 * 0.75          # reads row 5, at its fixed point
    Q[6, 2] = Mr[6, 2] = 2.0
    Ms[6, 2], Mt[6, 2] = 24, 1                                     # reads an all-zero row
    return [(5, 1), (8, 0), (6, 2), (5, 1), (8, 0)]


def case_null_after_change(st):
    Mr, Ms, Mt = st['Mr'], st['Ms'], st['Mt']
    Mr[3, 1] = 1.0                                                # changes Q[3,1]
    Ms[7, 2], Mt[7, 2] = 3, 1                                     # null on the pre-batch table, not in order
    return [(3, 1), (7, 2)]


def case_chains(st):
    Mr, Ms, Mt = st['Mr'], st['Ms'], st['Mt']
    Mr[3, 1] = 1.0
    for s, a, s2 in [(7, 2, 3), (9, 0, 7), (11, 3, 9), (14, 1, 11), (16, 2, 14)]:
        Ms[s, a], Mt[s, a] = s2, 1                                # each reads the row the previous one writes
    for s, a, s2 in [(18, 1, 15), (20, 3, 18), (21, 0, 20)]:
        Ms[s, a], Mt[s, a] = s2, 1                                # reads of rows written by null updates only
    Mr[21, 0] = 0.5                                               # ... and one of them changes
    return [(3, 1), (7, 2), (9, 0), (15, 0), (11, 3), (18, 1), (14, 1), (20, 3), (16, 2), (21, 0)]


def case_write_after_read(st):
    Q, Mr, Ms, Mt = st['Q'], st['Mr'], st['Ms'], st['Mt']
    Ms[20, 0], Mt[20, 0] = 21, 1
    Q[21, :2] = 0.5, 0.25                                         # (20,0) reads row 21 ...
    Mr[21, 0] = 2.0                                               # ... which (21,0) then changes
    Ms[4, 0], Mt[4, 0] = 6, 1                                     # a null reader of row 6 ...
    Mr[6, 0] = 1.0                                                # ... before (6,0) changes it
    Mr[22, 1] = 1.0
    Ms[23, 0], Mt[23, 0] = 22, 1
    return [(20, 0), (4, 0), (21, 0), (22, 1), (6, 0), (23, 0), (20, 0)]


def case_duplicates(st):
    Mr, Ms, Mt = st['Mr'], st['Ms'], st['Mt']
    Mr[18, 3] = 1.0
    Ms[13, 1], Mt[13, 1] = 18, 1
    return [(18, 3), (10, 0), (18, 3), (13, 1), (10, 0), (18, 3), (13, 1), (10, 0), (18, 3)]


def case_signed_zeros(st):
    Q, Mr, Ms, Mt = st['Q'], st['Mr'], st['Ms'], st['Mt']
    Q[1, 0] = -0.0                                                # Q + lr*0 = +0.0: equal, not the same bits
    Q[2, :] = -0.0
    Ms[5, 3], Mt[5, 3], Q[5, 3] = 2, 1, 0.0                       # max over a row of -0.0
    Q[9, :] = -0.25, -0.5, -1.0, -0.0
    Ms[10, 2], Mt[10, 2], Mr[10, 2], Q[10, 2] = 9, 1, -0.5, -0.0
    Mr[3, 2] = -0.5                                               # negative reward
    Ms[8, 1], Mt[8, 1] = 3, 1                                     # reads the row (3,2) writes
    return [(1, 0), (5, 3), (3, 2), (10, 2), (8, 1), (2, 1), (1, 0)]


CASES = [case_all_null, case_null_after_change, case_chains, case_write_after_read, case_duplicates,
         case_signed_zeros]


def classify(st, idx):
    """Per update of one batch of <= 32: null (the speculative value on the pre-batch table has the bits of
    Q[s,a]), valid (every earlier update writing what it reads is valid and null) and numerically unchanged."""
    Q, Mr, Ms, Mt = st['Q'], st['Mr'], st['Ms'], st['Mt']
    null, valid, same = [], [], []
    for j, i in enumerate(idx):
        s, a = divmod(i, A)
        s2 = int(Ms[s, a])
        td = Mr[s, a]
        td += GAMMA * int(Mt[s, a]) * np.amax(Q[s2])
        td -= Q[s, a]
        y = Q[s, a] + LR * td
        null.append(bits(y) == bits(Q[s, a]))
        same.append(y == Q[s, a])
        valid.append(all(valid[k] and null[k] for k in range(j) if idx[k] // A == s2 or idx[k] == i))
    return np.array(null), np.array(valid), np.array(same)


def layout(case, batch, rng):
    """Preset tables and this agent's uniforms: draw 0 (environment constructor), the reset to START, the action
    draw, the deliberate first replay batch, then random draws for the later steps."""
    st = tb.dynaq_init(S, A)
    lanes = case(st)
    full = (lanes + FILLER * 4)[:32]
    idx = (full + lanes[:1])[:batch]                               # a batch of 33 ends with a single changing update
    starts = list(tb.compile_gridworld(world())['starts'])
    head = [0.5, (starts.index(START) + 0.5) / len(starts), 0.1] + [(s * A + a + 0.5) / (S * A) for s, a in idx]
    u = np.concatenate([head, rng.random(4000)])
    return st, [s * A + a for s, a in idx], u


def run_cuda(presets, u, trials, steps, batch):
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import DynaQ
    from cobel_rl_b200.policy import EpsilonGreedy
    n = len(presets)
    stream = cb.BatchStream(n, device='cuda:0', user_stream=u)
    env = Gridworld(world(), rng=stream)
    ag = DynaQ(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream))
    for name, t in (('Q', ag._Q), ('Mr', ag.M._rewards), ('Ms', ag.M._states), ('Mt', ag.M._terminals)):
        t.copy_(torch.as_tensor(np.stack([p[name] for p in presets])).to(t.dtype))
    ag.record = True
    res = ag.train(env, trials, steps, batch)
    torch.cuda.synchronize()
    tables = {'Q': ag._Q.cpu().numpy(), 'Mr': ag.M._rewards.cpu().numpy(), 'Ms': ag.M._states.cpu().numpy(),
              'Mt': ag.M._terminals.cpu().numpy()}
    return res, tables, stream.draw_count.cpu().numpy()


def assert_agent(res, tables, draws, i, st, rec, k, what):
    W = tb.compile_gridworld(world())
    got = unpack_run(res, i, A, W['succ'], W['reward'])
    for key in ('states', 'actions', 'trial_steps', 'replay'):
        assert np.array_equal(got[key], rec[key]), '%s: %s differs' % (what, key)
    for key in ('Q', 'Mr'):                                       # bit for bit: -0.0 is not +0.0
        assert np.array_equal(bits(tables[key][i]), bits(st[key])), '%s: %s differs' % (what, key)
    assert np.array_equal(tables['Ms'][i], st['Ms']) and np.array_equal(tables['Mt'][i], st['Mt']), what
    assert int(draws[i]) == k, what


@pytest.mark.parametrize('batch', [7, 32, 33])
def test_deliberate_batches_match_the_oracle(batch):
    W = tb.compile_gridworld(world())
    rng = np.random.default_rng(batch)
    trials, steps = 2, 4
    built = [layout(c, batch, rng) for c in CASES]
    res, tables, draws = run_cuda([b[0] for b in built], np.stack([b[2] for b in built]), trials, steps, batch)
    for i, (case, (st, idx, u)) in enumerate(zip(CASES, built)):
        # the first replay batch is what the case says it is
        pre = {k: v.copy() for k, v in st.items()}
        tb.dynaq_train(W, pre, tb.Draws(u, 1), 1, 1, 0)           # the first step without its replay
        null, valid, same = classify(pre, idx[:32])
        after = {k: v.copy() for k, v in pre.items()}
        for i2 in idx[:32]:
            s, a = divmod(i2, A)
            tb._td_update(after['Q'], s, a, after['Mr'][s, a], int(after['Ms'][s, a]), int(after['Mt'][s, a]),
                          LR, GAMMA)
        changed = bits(after['Q']) != bits(pre['Q'])
        lost = [j for j in range(len(null)) if null[j] and not valid[j]]
        if batch >= 32:
            if case is case_all_null:
                assert null.all() and not changed.any()
            elif case is case_null_after_change:
                assert lost == [1] and changed[7, 2]                # dropping every null update loses this one
            elif case is case_chains:
                assert lost == [1, 2, 4, 6, 8] and all(changed[divmod(idx[j], A)] for j in lost)
                assert (null & valid)[[3, 5, 7]].all() and not null[9]
            elif case is case_write_after_read:
                assert not null[0] and not null[2] and null[1] and valid[1]
            elif case is case_duplicates:
                assert (~null).sum() == 4 and lost == [3, 6]
            elif case is case_signed_zeros:
                assert (same & ~null)[[0, 5, 6]].all() and (after['Mr'] < 0).any()
        # whole run against the sequential oracle
        rng_o = tb.Draws(u, 1)
        rec = tb.dynaq_train(W, st, rng_o, trials, steps, batch).arrays()
        assert_agent(res, tables, draws, i, st, rec, rng_o.k, '%s, batch %d' % (case.__name__, batch))


@pytest.mark.parametrize('batch', [7, 32, 33])
def test_random_batches_on_signed_zero_tables_match_the_oracle(batch):
    """Longer runs from tables with -0.0 entries and negative rewards, uniform replay draws."""
    W = tb.compile_gridworld(world())
    rng = np.random.default_rng(100 + batch)
    presets, us = [], []
    for g in range(3):
        st = tb.dynaq_init(S, A)
        st['Q'][rng.random((S, A)) < 0.5] = -0.0
        st['Mr'][:] = np.where(rng.random((S, A)) < 0.2, -0.25 * (g + 1), 0.0)
        st['Mt'][:] = (rng.random((S, A)) < 0.5).astype(np.int32)
        presets.append(st)
        us.append(rng.random(5000))
    trials, steps = 6, 20
    res, tables, draws = run_cuda(presets, np.stack(us), trials, steps, batch)
    for i, st in enumerate(presets):
        rng_o = tb.Draws(us[i], 1)
        rec = tb.dynaq_train(W, st, rng_o, trials, steps, batch).arrays()
        assert_agent(res, tables, draws, i, st, rec, rng_o.k, 'agent %d, batch %d' % (i, batch))


def test_pair_kernel_with_a_half_empty_last_warp_matches_the_oracle():
    """16385 agents: two agents per warp; the last agent shares its warp with an idle half."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import DynaQ
    from cobel_rl_b200.policy import EpsilonGreedy
    n, trials, steps, seed = 16385, 12, 50, 0xA11
    st0 = tb.dynaq_init(S, A)
    st0['Q'][::3, 1] = -0.0
    st0['Mr'][7, :] = -0.5
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    env = Gridworld(world(), rng=stream)
    ag = DynaQ(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream))
    ag._Q.copy_(torch.as_tensor(st0['Q']).expand_as(ag._Q))
    ag.M._rewards.copy_(torch.as_tensor(st0['Mr']).expand_as(ag.M._rewards))
    res = ag.train(env, trials, steps, 32)
    torch.cuda.synchronize()
    W = tb.compile_gridworld(world())
    Q, Mr = ag._Q.cpu().numpy(), ag.M._rewards.cpu().numpy()
    Ms, Mt = ag.M._states.cpu().numpy(), ag.M._terminals.cpu().numpy()
    for i in (0, 1, 8191, 16383, 16384):
        st = {k: v.copy() for k, v in st0.items()}
        rng = tb.Draws(LazyStream(seed, i), 1)
        rec = tb.dynaq_train(W, st, rng, trials, steps, 32).arrays()
        assert int(res['n_steps'][i]) == len(rec['states']), i
        assert np.array_equal(res['trial_steps'][i].cpu().numpy(), rec['trial_steps']), i
        assert np.array_equal(bits(Q[i]), bits(st['Q'])) and np.array_equal(bits(Mr[i]), bits(st['Mr'])), i
        assert np.array_equal(Ms[i], st['Ms']) and np.array_equal(Mt[i], st['Mt']), i
        assert int(stream.draw_count[i]) == rng.k, i
