"""Cost of recording replay_td: train() passes on two builds, alternated in one session.

    python profiles/replay_td.py --trees OLD_TREE NEW_TREE [--runs 3] [--workloads c2 c4 c3 c3g p20 p20r]

Every (run, tree, workload) is a process of its own that imports cobel_rl_b200 from that tree, trains a warm-up pass
and then PASSES timed passes, each on freshly initialised agents (host clock around train() and a device synchronise;
the construction of the agents is outside the window), so that a process times about half a second of train().  The
builds are alternated run by run so that both see the same machine state.  A build without the buffer (the parent of
the change) is the baseline.  In the recorded workloads (``agent.record = True``) both builds record step_sa,
step_next, step_td, replay_idx and replay_len; c3g and p20 do not record, and measure what the change costs a PMA call
that does not ask for replay_td in the generic kernels that store it: the one of every memory option and the one of
every world beyond 160 states (pma_main_kernel<4, false, BIG>, which has no PLAIN variant).  Prints the median pass of every process and a summary; the card's name and power
limit are read in the same session.

The horizons of C2 and C3 are shorter than the configurations' own: a recorded run holds 12 bytes per replayed update
(replay_idx and replay_td), which at C2's full 500 trials x 50 steps x 32 updates would be 39 GB.
  c2   4096 Dyna-Q agents, 5x5 open field, 250 trials x <=50 steps, batch 32 (config C2, half its trials), recorded
  c4   65536 SFMA agents, 20x20 open field, DR metric, default mode, 4 trials x <=200 steps, batch 32 (config C4),
       recorded
  c3   16384 PMA agents, 10x10 walled world, banded update_sr, 2 trials x <=100 steps, batch 32 (config C3, half its
       trials), recorded
  c3g  C3 not recorded, with M.ignore_barriers = False: the generic pma_main_kernel<4, false, false> (the PLAIN
       kernel is built for no memory option), as a call that does not ask for replay_td runs it
  p20  4096 PMA agents, walled 20x20 world (400 states), banded update_sr, 2 trials x <=100 steps, batch 32, not
       recorded
  p20r the same, recorded
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import time

SEED = 0x5EED
WALLS_10x10 = [(4, 5), (5, 4), (14, 15), (15, 14), (24, 25), (25, 24), (34, 35), (35, 34),
               (62, 72), (72, 62), (63, 73), (73, 63)]
WALLS_20x20 = [(5, 6), (6, 5), (25, 26), (26, 25), (45, 46), (46, 45), (208, 228), (228, 208), (209, 229), (229, 209)]
PASSES = {'c2': 50, 'c4': 10, 'c3': 16, 'c3g': 16, 'p20': 5, 'p20r': 5}    # timed passes per process, about 0.5 s in all


def child(tree, workload):
    sys.path.insert(0, tree)
    import numpy as np
    import torch
    import cobel_rl_b200 as cb
    from cobel_rl_b200 import agent as AG, memory as MEM
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.misc.gridworld_tools import make_gridworld, make_open_field
    from cobel_rl_b200.policy import EpsilonGreedy
    assert os.path.dirname(os.path.dirname(os.path.abspath(cb.__file__))) == os.path.abspath(tree)

    def make():
        if workload == 'c2':
            n, trials, steps = 4096, 250, 50
            world = make_gridworld(5, 5, terminals=[0], rewards=np.array([[0, 1]]), goals=[0])
        elif workload == 'c4':
            n, trials, steps = 65536, 4, 200
            world = make_open_field(20, 20, 0, 1)
        elif workload in ('p20', 'p20r'):
            n, trials, steps = 4096, 2, 100
            world = make_gridworld(20, 20, terminals=[19], rewards=np.array([[19, 10.0]]), goals=[19],
                                   starting_states=[210], invalid_transitions=WALLS_20x20)
        else:
            n, trials, steps = 16384, 2, 100
            world = make_gridworld(10, 10, terminals=[9], rewards=np.array([[9, 10]]), goals=[9], starting_states=[57],
                                   invalid_transitions=WALLS_10x10)
        st = cb.BatchStream(n, seed=SEED, device='cuda:0')
        env = Gridworld(world, rng=st)
        pol = EpsilonGreedy(0.1, rng=st)
        if workload == 'c2':
            mem = MEM.DynaQMemory(env.n_states, 4, 0.9, rng=st)
            ag = AG.DynaQ(env.observation_space, env.action_space, pol, None, 0.99, 0.99, mem)
        elif workload == 'c4':
            from cobel_rl_b200.memory.utils.metrics import DR
            mem = MEM.SFMAMemory(DR(world['width'], world['height'], world['sas'], 0.9, world['invalid_transitions']),
                                 env.n_states, 4, rng=st)
            ag = AG.SFMA(env.observation_space, env.action_space, pol, mem, None, 0.99, 0.99, rng=st)
            ag.mask_actions = True
        else:
            mem = MEM.PMAMemory(world['sas'], EpsilonGreedy(0.1, rng=st), 0.9, 0.9, 0.9, 0.99, rng=st)
            ag = AG.PMA(env.observation_space, env.action_space, pol, mem, None, 0.9, 0.99)
            ag.mask_actions = True
        if workload == 'c3g':
            mem.ignore_barriers = False
        ag.record = workload not in ('p20', 'c3g')
        torch.cuda.synchronize()
        return env, ag, trials, steps

    times = []
    for k in range(1 + PASSES[workload]):             # pass 0 warms up
        env, ag, trials, steps = make()
        t0 = time.perf_counter()
        res = ag.train(env, trials, steps, 32)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        replays = int(res['n_replay'].sum())
        has_td = 'replay_td' in res
        del res, ag, env
        gc.collect()                                    # the agent and its callbacks refer to each other
        torch.cuda.empty_cache()
    timed = sorted(times[1:])
    print(json.dumps({'tree': tree, 'workload': workload, 'seconds': timed[len(timed) // 2], 'min': timed[0],
                      'max': timed[-1], 'passes': len(timed), 'total': sum(timed), 'warmup_seconds': times[0],
                      'replayed_updates': replays, 'replay_td': has_td}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--trees', nargs=2, metavar=('OLD', 'NEW'))
    ap.add_argument('--runs', type=int, default=3)
    ap.add_argument('--workloads', nargs='+', default=list(PASSES), choices=list(PASSES))
    ap.add_argument('--child', nargs=2, metavar=('TREE', 'WORKLOAD'), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        child(*args.child)
        return
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    print('# GPU: %s' % q.stdout.strip().splitlines()[0] if q.returncode == 0 else '# GPU: nvidia-smi failed')
    results = {}
    label = dict(zip(args.trees, ('old', 'new')))
    for wl in args.workloads:
        for run in range(args.runs):
            for tree in args.trees:
                p = subprocess.run([sys.executable, os.path.abspath(__file__), '--child', tree, wl],
                                   capture_output=True, text=True)
                if p.returncode:
                    sys.exit('%s %s failed:\n%s' % (tree, wl, p.stderr[-3000:]))
                r = json.loads(p.stdout.strip().splitlines()[-1])
                print('%-4s run %d  %-3s median %.4f s [%.4f, %.4f] of %d passes (%.2f s)  (%d replayed updates per pass, '
                      'replay_td %s)' % (wl, run, label[tree], r['seconds'], r['min'], r['max'], r['passes'], r['total'],
                                         r['replayed_updates'], r['replay_td']), flush=True)
                results.setdefault((wl, tree), []).append(r['seconds'])
    print('# summary: seconds per pass, median [min, max] over the %d runs of the per-process medians' % args.runs)
    for wl in args.workloads:
        med = {}
        for tree in args.trees:
            t = sorted(results[(wl, tree)])
            med[tree] = t[len(t) // 2]
            print('%-4s  %-3s %.4f  [%.4f, %.4f]' % (wl, label[tree], med[tree], t[0], t[-1]))
        old, new = (med[t] for t in args.trees)
        print('%-4s  new / old = %.3f' % (wl, new / old))


if __name__ == '__main__':
    main()
