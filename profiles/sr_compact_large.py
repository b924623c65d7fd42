#!/usr/bin/env python
"""Rates of the compact SR agent on visited sets beyond shared memory (sr_compact_large_kernel).

1. 60x60 open field, identical inputs: the dense SR kernel (compact=False) and the HBM-resident compact path
   (max_visited = 3600).  Their trajectories must agree: per-trial steps and draw counts are asserted equal.
2. 100x100 open field, 128 agents, max_visited = 10000 (about 102 GB of SRc), eps = 0.3, 10 trials x 1000
   steps: agent-steps/s and the mean / largest number of visited states reached.

Times are CUDA events around one train() call after a warm-up call on separate agents.  Prints the card and
its power limit first.  Usage: python profiles/sr_compact_large.py [--agents 128] [--small-agents 32]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cobel_rl_b200 as cb  # noqa: E402
from cobel_rl_b200.agent import SR  # noqa: E402
from cobel_rl_b200.interface import Gridworld  # noqa: E402
from cobel_rl_b200.misc.gridworld_tools import make_open_field  # noqa: E402
from cobel_rl_b200.policy import EpsilonGreedy  # noqa: E402


def timed_train(world, n, seed, eps, trials, steps, **sr_kw):
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    env = Gridworld(world, rng=stream)
    ag = SR(env.observation_space, env.action_space, EpsilonGreedy(eps, rng=stream), None, 0.1, 0.95, **sr_kw)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    res = ag.train(env, trials, steps)
    t1.record()
    torch.cuda.synchronize()
    sec = t0.elapsed_time(t1) / 1e3
    agent_steps = int(res['n_steps'].sum())
    out = {'seconds': sec, 'agent_steps': agent_steps, 'agent_steps_per_s': agent_steps / sec,
           'trial_steps': res['trial_steps'].cpu(), 'draws': stream.draw_count.cpu().clone()}
    if sr_kw.get('compact'):
        out['n_visited_mean'] = float(ag.n_visited.double().mean())
        out['n_visited_max'] = int(ag.n_visited.max())
    del ag, env, stream, res
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--agents', type=int, default=128)
    ap.add_argument('--small-agents', type=int, default=32)
    args = ap.parse_args()
    print(subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv'], capture_output=True,
                         text=True).stdout.strip())
    report = {}

    w60 = make_open_field(60, 60, 0, 1, dense_sas=False)
    n = args.small_agents
    timed_train(w60, 2, 1, 0.3, 1, 50)                                        # warm-up: dense kernel
    timed_train(w60, 2, 1, 0.3, 1, 50, compact=True, max_visited=3600)      # warm-up: HBM compact kernel
    dense = timed_train(w60, n, 7, 0.3, 10, 500)
    large = timed_train(w60, n, 7, 0.3, 10, 500, compact=True, max_visited=3600)
    assert torch.equal(dense['trial_steps'], large['trial_steps']), 'trajectories differ'
    assert torch.equal(dense['draws'], large['draws']), 'draw counts differ'
    report['60x60'] = {'agents': n, 'trials': 10, 'steps': 500,
                       'dense_agent_steps_per_s': dense['agent_steps_per_s'],
                       'compact_hbm_agent_steps_per_s': large['agent_steps_per_s'],
                       'agent_steps': large['agent_steps'], 'n_visited_mean': large['n_visited_mean'],
                       'n_visited_max': large['n_visited_max']}
    print(json.dumps({'60x60': report['60x60']}), flush=True)

    w100 = make_open_field(100, 100, 0, 1, dense_sas=False)
    timed_train(w100, 2, 1, 0.3, 1, 50, compact=True, max_visited=10000)    # warm-up
    big = timed_train(w100, args.agents, 11, 0.3, 10, 1000, compact=True, max_visited=10000)
    report['100x100'] = {'agents': args.agents, 'trials': 10, 'steps': 1000, 'max_visited': 10000,
                         'seconds': big['seconds'], 'agent_steps': big['agent_steps'],
                         'agent_steps_per_s': big['agent_steps_per_s'], 'n_visited_mean': big['n_visited_mean'],
                         'n_visited_max': big['n_visited_max']}
    print(json.dumps({'100x100': report['100x100']}), flush=True)


if __name__ == '__main__':
    main()
