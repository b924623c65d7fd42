#!/usr/bin/env python
"""Rates of the compact SR agent's stand-alone methods (cobel_sr_compact_op, sr_compact_op_kernel).

100x100 open field, 128 agents, max_visited = 10000 (about 102 GB of SRc), trained eps = 0.3 for 10 trials x 1000
steps first (the visited sets then hold a few thousand states each, see profiles/sr_compact_large.py):
1. predict_on_batch(range(10000)): the value map of every agent, one launch; seconds per call and Q rows per second.
2. a hand-written step for all agents: retrieve_q + policy.select_action + env.step + update, in agent-steps/s, and
   the two SR calls alone (retrieve_q + update from fixed experiences).

Times are CUDA events around R calls after a warm-up; every call includes its Python side (argument checks,
one host synchronisation each for the state range check and, in update, the overflow flag).  Prints the card and its
power limit first.  Usage: python profiles/sr_compact_ops.py [--agents 128] [--reps 20] [--steps 200]"""
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


def timed(fn, reps):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--agents', type=int, default=128)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--steps', type=int, default=200)
    args = ap.parse_args()
    print(subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv'], capture_output=True,
                         text=True).stdout.strip())
    n, S = args.agents, 10000
    stream = cb.BatchStream(n, seed=11, device='cuda:0')
    env = Gridworld(make_open_field(100, 100, 0, 1, dense_sas=False), rng=stream)
    pol = EpsilonGreedy(0.3, rng=stream)
    ag = SR(env.observation_space, env.action_space, pol, None, 0.1, 0.95, compact=True, max_visited=S)
    ag.train(env, 10, 1000)
    torch.cuda.synchronize()
    report = {'agents': n, 'max_visited': S, 'n_visited_mean': float(ag.n_visited.double().mean()),
              'n_visited_max': int(ag.n_visited.max()),
              'reward_columns_max': int((ag.rewards != 0).sum(dim=1).max())}

    states = range(S)
    ag.predict_on_batch(states)                                             # warm-up
    sec = timed(lambda: ag.predict_on_batch(states), args.reps) / args.reps
    report['predict_on_batch_10000'] = {'seconds_per_call': sec, 'q_rows_per_s': n * S / sec}
    print(json.dumps(report), flush=True)

    state, _ = env.reset()

    def step():
        nonlocal state
        action = pol.select_action(ag.retrieve_q(state))
        nxt, reward, end, _trunc, _info = env.step(action)
        ag.update({'state': state, 'action': action, 'reward': reward, 'next_state': nxt, 'terminal': 1 - end.int()})
        state = nxt

    for _ in range(10):                                                     # warm-up
        step()
    sec = timed(step, args.steps)
    s0 = state.clone()
    exp = {'state': s0, 'action': 0, 'reward': 0.0, 'next_state': s0, 'terminal': 1}

    def ops():
        ag.retrieve_q(s0)
        ag.update(exp)
    ops()
    sec_ops = timed(ops, args.steps)
    report['hand_written_step'] = {'steps': args.steps, 'agent_steps_per_s': n * args.steps / sec,
                                   'seconds_per_step': sec / args.steps,
                                   'retrieve_q_plus_update_agent_steps_per_s': n * args.steps / sec_ops,
                                   'retrieve_q_plus_update_seconds': sec_ops / args.steps}
    print(json.dumps({'hand_written_step': report['hand_written_step']}), flush=True)


if __name__ == '__main__':
    main()
