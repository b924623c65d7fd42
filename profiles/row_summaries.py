"""How often dynaq_warp_kernel<A, PLAIN, false, SUM> refreshes its row summaries, and a check that they stay exact
(DESIGN.md K1).  CPU only: the oracle's Dyna-Q loop on the bench's C2 setting (5x5 open field, 500 trials x <= 50
steps, batch 32, the bench's seed and per-agent streams), run twice side by side: once in the reference's order and
once as the summary kernel computes it:

  * the action is drawn from the tie pattern P[s], not from row Q[s,:];
  * the online update's target reads V[s2]; when the update changes Q[s,a] (bitwise) V[s] and P[s] are rebuilt
    from the row ("online refresh");
  * the replay's speculative pass reads V[s2_j]; the kept updates run in the kernel's dependency rounds on full rows,
    the first round committing the speculative values; after the last round every kept lane rebuilds V and P of its
    state ("batch refresh").

After every step the tables and the stream position must be bit-identical in both runs, and V / P must equal the row
maximum and tie pattern recomputed from Q.

  python profiles/row_summaries.py [agent ...]        (default: agents 0 1; seconds per agent)
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from oracle import tabular as tb  # noqa: E402
from oracle.philox import LazyStream  # noqa: E402
from cobel_rl_b200.misc.gridworld_tools import make_gridworld  # noqa: E402
from step_overlap import BATCH, EPS, GAMMA, LR, MEM_LR, SEED, bits, rounds, td_value  # noqa: E402

CASES = ('steps', 'online_refresh', 'online_self_loop', 'max_changed', 'pattern_changed', 'nonnull_batches',
         'kept_lanes', 'refreshed_states', 'round_same_state')


def xmax(a, b):
    return b if a < b else a


def row_max(row):
    """row_max<A> (csrc/common.cuh): the kernel's compare-and-select order, whose pick between -0.0 and +0.0 may
    differ from np.amax's."""
    if len(row) == 4:
        return xmax(xmax(row[0], row[1]), xmax(row[2], row[3]))
    m = row[0]
    for x in row[1:]:
        m = xmax(m, x)
    return m


def summary(row):
    m = row_max(row)
    return m, sum(1 << a for a in range(len(row)) if row[a] == m)


def summary_step(W, st, V, P, s, step, steps, rng, n):
    """One step of the summary kernel's order from state s.  Returns (s2, fin)."""
    S, A = W['S'], W['A']
    Q, Mr, Ms, Mt = st['Q'], st['Mr'], st['Ms'], st['Mt']
    pattern = np.array([(P[s] >> x) & 1 for x in range(A)], dtype=np.float64)   # same tie set as row Q[s,:]
    a = tb.draw_categorical(tb.action_probs(('eps', EPS), pattern), rng.next())
    s2, r, end = tb.env_step(W, s, a)
    nt, fin = 1 - end, bool(end or step + 1 == steps)
    Mr[s, a] += MEM_LR * (r - Mr[s, a]); Ms[s, a] = s2; Mt[s, a] = nt
    q = Q[s, a]
    td = r
    td += GAMMA * nt * V[s2]
    td -= q
    qn = q + LR * td
    Q[s, a] = qn
    if bits(qn) != bits(q):
        n['online_refresh'] += 1
        n['online_self_loop'] += s2 == s
        m, p = summary(Q[s])
        n['max_changed'] += bits(m) != bits(V[s])
        n['pattern_changed'] += p != P[s]
        V[s], P[s] = m, p
    # replay: speculative pass on V, rounds on full rows, then the kept lanes' refresh
    items, spec, null = [], [], []
    for i in [tb.draw_integer(rng.next(), S * A) for _ in range(BATCH)]:
        rs, ra = divmod(i, A)
        items.append((rs, ra, int(Ms[rs, ra])))
        spec.append(td_value(np.array([V[items[-1][2]]]), Q[rs, ra], Mr[rs, ra], Mt[rs, ra]))
        null.append(bits(spec[-1]) == bits(Q[rs, ra]))
    if not all(null):
        valid = []
        for j, (rs, ra, x2) in enumerate(items):
            valid.append(all(valid[i] and null[i] for i in range(j)
                             if items[i][0] == x2 or items[i][:2] == (rs, ra)))
        kept = [not (v and z) for v, z in zip(valid, null)]
        for d, lanes in enumerate(rounds(items, kept)):
            states = [items[j][0] for j in lanes]
            n['round_same_state'] += len(states) - len(set(states))
            vals = [spec[j] if d == 0 else td_value(Q[items[j][2]], Q[items[j][0], items[j][1]],
                                                    Mr[items[j][0], items[j][1]], Mt[items[j][0], items[j][1]])
                    for j in lanes]
            for j, v in zip(lanes, vals):
                Q[items[j][0], items[j][1]] = v
        refreshed = {items[j][0] for j in range(BATCH) if kept[j]}
        n['nonnull_batches'] += 1
        n['kept_lanes'] += sum(kept)
        n['refreshed_states'] += len(refreshed)
        for x in refreshed:
            V[x], P[x] = summary(Q[x])
    n['steps'] += 1
    return s2, fin


def run(W, seed, agent, trials, steps, n=None, k0=1, Q0=None):
    """Both orders side by side for one agent whose stream starts at draw k0 (draw 0 goes to the environment's
    constructor), from the table Q0 (default zeros); asserts bit-identity and exact summaries after every step.
    Returns the case counts and the summary run's final tables and draw count."""
    n = n if n is not None else dict.fromkeys(CASES, 0)
    S, A = W['S'], W['A']
    ref, sm = tb.dynaq_init(S, A), tb.dynaq_init(S, A)
    if Q0 is not None:
        ref['Q'][:], sm['Q'][:] = Q0, Q0
    V = np.zeros(S)
    P = np.zeros(S, dtype=np.int64)
    for x in range(S):
        V[x], P[x] = summary(sm['Q'][x])
    rr, rk = tb.Draws(LazyStream(seed, agent), k0), tb.Draws(LazyStream(seed, agent), k0)
    for _ in range(trials):
        s = tb.env_reset(W, rr)
        assert tb.env_reset(W, rk) == s
        for step in range(steps):
            # the reference's order (tb.dynaq_train's step)
            a = tb.select_action(('eps', EPS), ref['Q'][s], None, rr)
            s2, r, end = tb.env_step(W, s, a)
            ref['Mr'][s, a] += MEM_LR * (r - ref['Mr'][s, a]); ref['Ms'][s, a] = s2; ref['Mt'][s, a] = 1 - end
            tb._td_update(ref['Q'], s, a, r, s2, 1 - end, LR, GAMMA)
            for i in [tb.draw_integer(rr.next(), S * A) for _ in range(BATCH)]:
                rs, ra = divmod(i, A)
                tb._td_update(ref['Q'], rs, ra, ref['Mr'][rs, ra], int(ref['Ms'][rs, ra]), int(ref['Mt'][rs, ra]),
                              LR, GAMMA)
            # the summary kernel's order
            s2k, fin = summary_step(W, sm, V, P, s, step, steps, rk, n)
            assert s2k == s2 and fin == bool(end or step + 1 == steps)
            assert rk.k == rr.k, 'draw count'
            for key in ('Q', 'Mr', 'Ms', 'Mt'):
                x, y = ref[key], sm[key]
                assert ((x.view(np.int64) == y.view(np.int64)) if x.dtype == np.float64 else (x == y)).all(), key
            for x in range(S):
                m, p = summary(sm['Q'][x])
                assert bits(V[x]) == bits(m) and P[x] == p, 'summary of state %d' % x
            s = s2
            if fin:
                break
    return n, sm, rk.k


def main():
    agents = [int(x) for x in sys.argv[1:]] or [0, 1]
    world = tb.compile_gridworld(make_gridworld(5, 5, terminals=[0], rewards=np.array([[0, 1]]), goals=[0]))
    n = dict.fromkeys(CASES, 0)
    for g in agents:
        run(world, SEED, g, 500, 50, n)
    st, nb = n['steps'], max(n['nonnull_batches'], 1)
    print('agents %s: %d steps, every step bit-identical to the sequential order, V and P exact after each' %
          (agents, st))
    print('  online refreshes (Q[s,a] changed)          %.4f per step (%d; %d self-loops s2 == s)' %
          (n['online_refresh'] / st, n['online_refresh'], n['online_self_loop']))
    print('    of which the row maximum changed         %d, the tie pattern changed %d' %
          (n['max_changed'], n['pattern_changed']))
    print('  batches with a kept update                 %.1f %% of steps' % (100 * n['nonnull_batches'] / st))
    print('    kept lanes per such batch                %.2f' % (n['kept_lanes'] / nb))
    print('    distinct refreshed states per batch      %.2f' % (n['refreshed_states'] / nb))
    print('  round lanes writing a state another lane of the round writes  %d' % n['round_same_state'])


if __name__ == '__main__':
    main()
