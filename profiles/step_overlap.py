"""How often the overlapped Dyna-Q step of dynaq_warp_kernel<A, PLAIN> takes each of its exact fix-ups, and a check
that the overlapped order gives the sequential result bit for bit (DESIGN.md K1).  CPU only: the oracle's Dyna-Q loop
on the bench's C2 setting (5x5 open field, 500 trials x <= 50 steps, batch 32, the bench's seed and per-agent
streams), run twice side by side: once in the reference's order and once in the kernel's order:

  * the replay gather (index, Mr, Ms, Mt) reads M before the step's store; a lane whose index is (s,a) takes the
    stored values ("gather fix-up");
  * the online update and the replay's speculative pass read Q before the online write; a replay lane whose entry is
    Q[s,a] ("entry substitution") or whose max row is Q[s,:] ("row substitution") takes the online result qn;
  * the next action is selected from Q[s2,:] (element a = qn when s2 == s) and the draw after the replay's 32 before
    the replay is applied; it stands when no kept replay update writes row s2, else it is selected again;
  * the replay keeps the updates that are not valid-and-null and applies them in the kernel's dependency rounds, the
    first round committing the speculative values.

After every step the tables, the next action and the stream position must be bit-identical in both runs.

  python profiles/step_overlap.py [agent ...]        (default: agents 0 1; seconds per agent)
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
BATCH = 32
CASES = ('steps', 'gather_fixup', 'entry_subst', 'row_subst', 'reads_qsa', 'online_null', 'all_null',
         'action_kept_null', 'action_kept_ballot', 'action_recomputed', 'action_changed', 'trial_end')


def bits(x):
    return np.float64(x).view(np.int64)


def td_value(row, q, r, nt):
    """_td_update's value without the write (agent/dyna_q.py:275-301)."""
    td = r
    td += GAMMA * nt * np.amax(row)
    td -= q
    return q + LR * td


def rounds(items, keep):
    """The kernel's dependency rounds over the kept updates: lists of lane indices, in order."""
    lvl = {}
    for j, (s, a, s2) in enumerate(items):
        if keep[j]:
            lvl[j] = 1 + max([lvl[i] for i in lvl if items[i][0] == s2 or items[i][:2] == (s, a) or
                              items[i][2] == s], default=0)
    return [[j for j in lvl if lvl[j] == d] for d in range(1, max(lvl.values(), default=0) + 1)]


def overlapped_step(W, st, s, a, step, steps, rng, n):
    """One step of the kernel's order from (s, a), the action draw already taken.  Returns (s2, r, fin, a2)."""
    S, A = W['S'], W['A']
    Q, Mr, Ms, Mt = st['Q'], st['Mr'], st['Ms'], st['Mt']
    s2, r, end = tb.env_step(W, s, a)
    nt, fin, sa = 1 - end, bool(end or step + 1 == steps), s * A + a
    # gather before the store
    idx = [tb.draw_integer(rng.u[rng.k + j], S * A) for j in range(BATCH)]
    rr = [Mr.flat[i] for i in idx]
    rs2 = [int(Ms.flat[i]) for i in idx]
    rnt = [int(Mt.flat[i]) for i in idx]
    # store + online update against the table before either write
    m1 = Mr[s, a] + MEM_LR * (r - Mr[s, a])
    qn = td_value(Q[s2], Q[s, a], r, nt)
    n['online_null'] += bits(qn) == bits(Q[s, a])
    # next action, speculatively
    a2 = None
    if not fin:
        row = Q[s2].copy()
        if s2 == s:
            row[a] = qn
        a2 = tb.draw_categorical(tb.action_probs(('eps', EPS), row), rng.u[rng.k + BATCH])
    # gather fix-up and the speculative pass with the substitutions
    items, spec, null = [], [], []
    for j, i in enumerate(idx):
        if i == sa:
            rr[j], rs2[j], rnt[j] = m1, s2, nt
            n['gather_fixup'] += 1
        rs, ra = divmod(i, A)
        row = Q[rs2[j]].copy()
        if rs2[j] == s:
            row[a] = qn
            n['row_subst'] += 1
        q = qn if i == sa else Q[rs, ra]
        n['entry_subst'] += i == sa
        n['reads_qsa'] += i == sa or rs2[j] == s
        items.append((rs, ra, rs2[j]))
        spec.append(td_value(row, q, rr[j], rnt[j]))
        null.append(bits(spec[-1]) == bits(q))
    # the online write, then the replay
    Mr[s, a], Ms[s, a], Mt[s, a], Q[s, a] = m1, s2, nt, qn
    kept = [False] * BATCH
    if all(null):
        n['all_null'] += 1
    else:
        valid = []
        for j, (rs, ra, x2) in enumerate(items):
            valid.append(all(valid[i] and null[i] for i in range(j)
                             if items[i][0] == x2 or items[i][:2] == (rs, ra)))
        kept = [not (v and z) for v, z in zip(valid, null)]
        for d, lanes in enumerate(rounds(items, kept)):
            vals = [spec[j] if d == 0 else td_value(Q[items[j][2]], Q[items[j][0], items[j][1]], rr[j], rnt[j])
                    for j in lanes]
            for j, v in zip(lanes, vals):
                Q[items[j][0], items[j][1]] = v
    rng.k += BATCH
    if fin:
        n['trial_end'] += 1
    elif all(null):
        n['action_kept_null'] += 1
    elif not any(k and it[0] == s2 for k, it in zip(kept, items)):
        n['action_kept_ballot'] += 1
    else:
        n['action_recomputed'] += 1
        old = a2
        a2 = tb.draw_categorical(tb.action_probs(('eps', EPS), Q[s2]), rng.u[rng.k])
        n['action_changed'] += old != a2
    if not fin:
        rng.k += 1
    n['steps'] += 1
    return s2, r, fin, a2


def run(W, seed, agent, trials, steps, n=None, k0=1):
    """Both orders side by side for one agent whose stream starts at draw k0 (draw 0 goes to the environment's
    constructor); asserts bit-identity after every step.  Returns the case counts and the overlapped run's final
    tables and draw count."""
    n = n if n is not None else dict.fromkeys(CASES, 0)
    S, A = W['S'], W['A']
    ref, ovl = tb.dynaq_init(S, A), tb.dynaq_init(S, A)
    rr, ro = tb.Draws(LazyStream(seed, agent), k0), tb.Draws(LazyStream(seed, agent), k0)
    for _ in range(trials):
        s = tb.env_reset(W, rr)
        assert tb.env_reset(W, ro) == s
        a = tb.select_action(('eps', EPS), ovl['Q'][s], None, ro)
        for step in range(steps):
            # the reference's order (tb.dynaq_train's step)
            ar = tb.select_action(('eps', EPS), ref['Q'][s], None, rr)
            assert ar == a, 'action'
            s2, r, end = tb.env_step(W, s, ar)
            ref['Mr'][s, ar] += MEM_LR * (r - ref['Mr'][s, ar]); ref['Ms'][s, ar] = s2; ref['Mt'][s, ar] = 1 - end
            tb._td_update(ref['Q'], s, ar, r, s2, 1 - end, LR, GAMMA)
            for i in [tb.draw_integer(rr.next(), S * A) for _ in range(BATCH)]:
                rs, ra = divmod(i, A)
                tb._td_update(ref['Q'], rs, ra, ref['Mr'][rs, ra], int(ref['Ms'][rs, ra]), int(ref['Mt'][rs, ra]),
                              LR, GAMMA)
            # the kernel's order
            s2o, _, fin, a = overlapped_step(W, ovl, s, a, step, steps, ro, n)
            assert s2o == s2 and fin == bool(end or step + 1 == steps)
            for key in ('Q', 'Mr', 'Ms', 'Mt'):
                x, y = ref[key], ovl[key]
                assert ((x.view(np.int64) == y.view(np.int64)) if x.dtype == np.float64 else (x == y)).all(), key
            s = s2
            if fin:
                assert ro.k == rr.k, 'draw count'
                break
            assert ro.k == rr.k + 1, 'draw count'
    return n, ovl, ro.k


def main():
    agents = [int(x) for x in sys.argv[1:]] or [0, 1]
    world = tb.compile_gridworld(make_gridworld(5, 5, terminals=[0], rewards=np.array([[0, 1]]), goals=[0]))
    n = dict.fromkeys(CASES, 0)
    for g in agents:
        run(world, SEED, g, 500, 50, n)
    st = n['steps']
    print('agents %s: %d steps, every step bit-identical to the sequential order' % (agents, st))
    print('  replay lanes whose index is the stored (s,a)       %.3f per step (%.2f %% of lanes)' %
          (n['gather_fixup'] / st, 100 * n['gather_fixup'] / (st * BATCH)))
    print('  replay lanes that read Q[s,a] (entry or max row)   %.3f per step (entry %.3f, row %.3f)' %
          (n['reads_qsa'] / st, n['entry_subst'] / st, n['row_subst'] / st))
    print('  online updates that leave Q[s,a] bit-identical    %.1f %%' % (100 * n['online_null'] / st))
    print('  replay batches with all 32 updates null            %.1f %%' % (100 * n['all_null'] / st))
    nf = st - n['trial_end']
    print('  steps that select a next action                    %.1f %%  (the others end a trial)' % (100 * nf / st))
    print('    speculative action stands: all-null batch        %.1f %%' % (100 * n['action_kept_null'] / nf))
    print('    speculative action stands: row s2 not written    %.1f %%' % (100 * n['action_kept_ballot'] / nf))
    print('    selected again after the rounds                  %.1f %%  (a different action in %d steps)' %
          (100 * n['action_recomputed'] / nf, n['action_changed']))


if __name__ == '__main__':
    main()
