"""How many of the Dyna-Q replay's TD updates leave Q bit-identical, and how deep the replay's dependency graph is
with and without them (DESIGN.md K1).  CPU only: the oracle's Dyna-Q loop on the bench's C2 setting (5x5 open field,
500 trials x <= 50 steps, batch 32, the bench's seed and per-agent streams) with an instrumented replay.

For every replay batch of 32 it evaluates each update against the pre-batch table ("speculative"), marks it null
when the result has the bits of Q[s,a] and valid when every earlier update that writes what it reads (row Q[s2,:],
entry Q[s,a]) is valid and null, and checks that the sequential result without the valid null updates is
bit-identical to the full sequential result.  Rounds are the depth of the dependency graph under the kernel's rule
(i < j: i writes row s2_j or entry (s_j,a_j), or i reads row s_j).

  python profiles/replay_nulls.py [agent ...]        (default: agents 0 1; a few minutes per agent)
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import tabular as tb  # noqa: E402
from oracle.philox import LazyStream  # noqa: E402
from cobel_rl_b200.misc.gridworld_tools import make_gridworld  # noqa: E402

SEED = 0x5EED
LR, GAMMA, MEM_LR, EPS = 0.99, 0.99, 0.9, 0.1


def bits(x):
    return np.float64(x).view(np.int64)


def depth(items, keep):
    lvl, best = [0] * len(items), 0
    for j, (s, a, s2) in enumerate(items):
        if not keep[j]:
            continue
        lv = 1
        for i in range(j):
            si, ai, s2i = items[i]
            if keep[i] and (si == s2 or (si == s and ai == a) or s2i == s):
                lv = max(lv, lvl[i] + 1)
        lvl[j], best = lv, max(best, lv)
    return best


def run(W, agent, trials=500, steps=50, batch=32):
    """One row per replay batch: trial, null updates, all null, both 16-update halves all null, updates that
    change Q in sequential order, rounds today, rounds with the valid null updates dropped."""
    S, A = W['S'], W['A']
    st = tb.dynaq_init(S, A)
    Q, Mr, Ms, Mt = st['Q'], st['Mr'], st['Ms'], st['Mt']
    rng = tb.Draws(LazyStream(SEED, agent), 1)
    rows = []
    for trial in range(trials):
        s = tb.env_reset(W, rng)
        for _ in range(steps):
            a = tb.select_action(('eps', EPS), Q[s], None, rng)
            s2, r, end = tb.env_step(W, s, a, rng)
            Mr[s, a] += MEM_LR * (r - Mr[s, a]); Ms[s, a] = s2; Mt[s, a] = 1 - end
            tb._td_update(Q, s, a, r, s2, 1 - end, LR, GAMMA)
            s = s2
            idx = [tb.draw_integer(rng.next(), S * A) for _ in range(batch)]
            items = [(i // A, i % A, int(Ms[i // A, i % A])) for i in idx]
            Q0 = Q.copy()
            null, valid = [], []
            for j, (rs, ra, rs2) in enumerate(items):
                q = Q0[rs, ra]
                td = Mr[rs, ra]
                td += GAMMA * Mt[rs, ra] * np.amax(Q0[rs2])
                td -= q
                null.append(bits(q + LR * td) == bits(q))
                valid.append(all(valid[i] and null[i] for i in range(j)
                                 if items[i][0] == rs2 or (items[i][0] == rs and items[i][1] == ra)))
            keep = [not (v and n) for v, n in zip(valid, null)]
            changed = 0
            for rs, ra, rs2 in items:
                old = Q[rs, ra]
                tb._td_update(Q, rs, ra, Mr[rs, ra], rs2, int(Mt[rs, ra]), LR, GAMMA)
                changed += bits(Q[rs, ra]) != bits(old)
            Qp = Q0
            for k, (rs, ra, rs2) in zip(keep, items):
                if k:
                    tb._td_update(Qp, rs, ra, Mr[rs, ra], rs2, int(Mt[rs, ra]), LR, GAMMA)
            assert (Qp.view(np.int64) == Q.view(np.int64)).all(), 'dropping the valid null updates changed Q'
            rows.append((trial, sum(null), all(null), (all(null[:16]) + all(null[16:])) / 2, changed,
                         depth(items, [True] * batch), depth(items, keep)))
            if end:
                break
    return np.array(rows, dtype=float)


def main():
    agents = [int(x) for x in sys.argv[1:]] or [0, 1]
    world = make_gridworld(5, 5, terminals=[0], rewards=np.array([[0, 1]]), goals=[0])
    W = tb.compile_gridworld(world)
    o = np.concatenate([run(W, g) for g in agents])
    alln = o[:, 2] == 1
    print('agents %s: %d replay batches of 32' % (agents, len(o)))
    print('  null updates (pre-batch table)   %.2f / 32' % o[:, 1].mean())
    print('  batches with all 32 null         %.1f %%  (16-update halves: %.1f %%)' % (100 * alln.mean(),
                                                                                       100 * o[:, 3].mean()))
    print('  rounds per batch, all updates    %.2f' % o[:, 5].mean())
    print('  rounds, all-null batches skipped %.2f' % (o[:, 5] * ~alln).mean())
    print('  rounds, valid null dropped       %.2f  (%.2f in the batches with a change)' % (o[:, 6].mean(),
                                                                                          o[~alln, 6].mean()))
    for lo, hi in [(0, 10), (10, 50), (50, 500)]:
        m = (o[:, 0] >= lo) & (o[:, 0] < hi)
        print('  trials %3d-%3d: %5d batches, %.1f updates per batch change Q' % (lo, hi, m.sum(), o[m, 4].mean()))


if __name__ == '__main__':
    main()
