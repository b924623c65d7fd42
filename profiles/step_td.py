"""Cost of recording step_td: one train() pass with ``agent.record = True`` on two builds, alternated in one session.

    python profiles/step_td.py --trees OLD_TREE NEW_TREE [--runs 3] [--workloads c2 c4]

Every (run, tree, workload) is a process of its own that imports cobel_rl_b200 from that tree, trains a warm-up pass
and then one timed pass on freshly initialised agents (host clock around train() and a device synchronise; the
construction of the agents is outside the window).  The builds are alternated run by run so that both see the same
machine state.  There is no switch that turns step_td off while ``record`` is on: a build without the buffer (the
parent of the change) is the baseline.  Prints one line per pass and a summary; the card's name and power limit are
read in the same session.

  c2  4096 Dyna-Q agents, 5x5 open field, 500 trials x <=50 steps, batch 32 (config C2)
  c4  65536 SFMA agents, 20x20 open field, DR metric, default mode, 4 trials x <=200 steps, batch 32 (config C4)
"""
import argparse
import json
import os
import subprocess
import sys
import time

SEED = 0x5EED


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
            n, trials, steps = 4096, 500, 50
            world = make_gridworld(5, 5, terminals=[0], rewards=np.array([[0, 1]]), goals=[0])
        else:
            n, trials, steps = 65536, 4, 200
            world = make_open_field(20, 20, 0, 1)
        st = cb.BatchStream(n, seed=SEED, device='cuda:0')
        env = Gridworld(world, rng=st)
        pol = EpsilonGreedy(0.1, rng=st)
        if workload == 'c2':
            mem = MEM.DynaQMemory(env.n_states, 4, 0.9, rng=st)
            ag = AG.DynaQ(env.observation_space, env.action_space, pol, None, 0.99, 0.99, mem)
        else:
            from cobel_rl_b200.memory.utils.metrics import DR
            mem = MEM.SFMAMemory(DR(world['width'], world['height'], world['sas'], 0.9, world['invalid_transitions']),
                                 env.n_states, 4, rng=st)
            ag = AG.SFMA(env.observation_space, env.action_space, pol, mem, None, 0.99, 0.99, rng=st)
            ag.mask_actions = True
        ag.record = True
        torch.cuda.synchronize()
        return env, ag, trials, steps

    out = {}
    for label in ('warmup', 'timed'):
        env, ag, trials, steps = make()
        t0 = time.perf_counter()
        res = ag.train(env, trials, steps, 32)
        torch.cuda.synchronize()
        out[label] = time.perf_counter() - t0
        agent_steps = int(res['n_steps'].sum())
        has_td = 'step_td' in res
        del res, ag, env
        torch.cuda.empty_cache()
    print(json.dumps({'tree': tree, 'workload': workload, 'seconds': out['timed'], 'warmup_seconds': out['warmup'],
                      'agent_steps': agent_steps, 'step_td': has_td}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--trees', nargs=2, metavar=('OLD', 'NEW'))
    ap.add_argument('--runs', type=int, default=3)
    ap.add_argument('--workloads', nargs='+', default=['c2', 'c4'], choices=['c2', 'c4'])
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
                print('%s run %d  %-3s %8.3f s  (%d agent-steps, step_td %s)' % (
                    wl, run, label[tree], r['seconds'], r['agent_steps'], r['step_td']), flush=True)
                results.setdefault((wl, tree), []).append(r['seconds'])
    print('# summary: seconds per pass, median [min, max] of %d runs' % args.runs)
    for wl in args.workloads:
        med = {}
        for tree in args.trees:
            t = sorted(results[(wl, tree)])
            med[tree] = t[len(t) // 2]
            print('%s  %-3s %8.3f  [%.3f, %.3f]' % (wl, label[tree], med[tree], t[0], t[-1]))
        old, new = (med[t] for t in args.trees)
        print('%s  new / old = %.3f' % (wl, new / old))


if __name__ == '__main__':
    main()
