#!/usr/bin/env python
"""Times of PMA's stand-alone replay beyond 160 states (cobel_pma_replay, BIG branch of csrc/pma.cu replay_only).

The walled 20x20 world of tests/test_pma_gpu.py::test_pma_20x20_large_state_space (400 states, 1600 one-step
backups, half band 20), 4096 agents, trained fused for 3 trials x 100 steps first.  Then, per call:
1. replay(32, s), replay(32, s, update_sr=True) and compute_need(None);
2. one hand-written trial -- replay(start), `steps` steps of select_action + env.step + update_q + store for all agents,
   replay(None, update_sr=True) -- against one fused train() trial of the same length;
3. the host-side band re-measure that sr_band() makes after every store() (one pass over all of T), alone and as part
   of a replay call (with it, the call also runs pma_band_check_kernel).

Times are CUDA events around R calls after a warm-up; every call includes its Python side.  Prints the card and its
power limit first.  Usage: python profiles/pma_big_ops.py [--agents 4096] [--reps 10] [--steps 50]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cobel_rl_b200 as cb  # noqa: E402
from cobel_rl_b200.agent import PMA  # noqa: E402
from cobel_rl_b200.interface import Gridworld  # noqa: E402
from cobel_rl_b200.memory import PMAMemory  # noqa: E402
from cobel_rl_b200.misc import gridworld_tools as mg  # noqa: E402
from cobel_rl_b200.policy import EpsilonGreedy  # noqa: E402

WALLS = [(5, 6), (6, 5), (25, 26), (26, 25), (45, 46), (46, 45), (208, 228), (228, 208), (209, 229), (229, 209)]


def timed(fn, reps, setup=None):
    """Seconds per call of fn; `setup` runs before every call, outside the timed window."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    torch.cuda.synchronize()
    for t0, t1 in ev:
        if setup:
            setup()
        t0.record()
        fn()
        t1.record()
    torch.cuda.synchronize()
    return sum(t0.elapsed_time(t1) for t0, t1 in ev) / 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--agents', type=int, default=4096)
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--steps', type=int, default=50)
    args = ap.parse_args()
    print(subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv'],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    n, L = args.agents, 32
    world = mg.make_gridworld(20, 20, terminals=[19], rewards=np.array([[19, 10.0]]), goals=[19], starting_states=[210],
                              invalid_transitions=WALLS)
    stream = cb.BatchStream(n, seed=7, device='cuda:0')
    env = Gridworld(world, rng=stream)
    mem = PMAMemory(world['sas'], EpsilonGreedy(0.1, rng=stream), 0.9, 0.9, 0.9, 0.99, rng=stream)
    pol = EpsilonGreedy(0.1, rng=stream)
    ag = PMA(env.observation_space, env.action_space, pol, mem)
    ag.mask_actions = True
    ag.action_mask = torch.as_tensor(np.argmax(world['sas'], axis=2) != np.arange(400)[:, None])
    ag.train(env, 3, 100, L)
    torch.cuda.synchronize()
    report = {'agents': n, 'states': 400, 'band': mem.sr_band(env.transition_band)[0], 'replay_length': L}
    s = torch.arange(n, device='cuda:0') % 400

    calls = {'replay': lambda: ag.replay(L, s), 'replay_update_sr': lambda: ag.replay(L, s, update_sr=True),
             'replay_none': lambda: ag.replay(L, None), 'compute_need_none': lambda: mem.compute_need(None)}
    for name, fn in calls.items():
        fn()                                                                 # warm-up
        report[name + '_s'] = timed(fn, args.reps)
    print(json.dumps(report), flush=True)

    # band re-measure: what sr_band() does when store() has reset the cached band
    def forget():
        mem._band_T = None
    mem.sr_band(env.transition_band)
    report['band_remeasure_s'] = timed(lambda: mem.sr_band(env.transition_band), args.reps, forget)
    report['replay_after_store_s'] = timed(calls['replay'], args.reps, forget)
    report['replay_update_sr_after_store_s'] = timed(calls['replay_update_sr'], args.reps, forget)
    print(json.dumps({k: report[k] for k in ('band_remeasure_s', 'replay_after_store_s', 'replay_update_sr_after_store_s')}),
          flush=True)

    mask = ag.action_mask

    def hand_trial():
        state, _ = env.reset()
        ag.replay(L, state)
        for _ in range(args.steps):
            action = pol.select_action(ag.Q[torch.arange(n, device='cuda:0'), state], mask[state])
            nxt, reward, end, _trunc, _info = env.step(action)
            exp = {'state': state, 'action': action, 'reward': reward, 'next_state': nxt, 'terminal': 1 - end.int()}
            ag.update_q([exp])
            mem.store(exp)
            state = nxt
        ag.replay(L, None, update_sr=True)

    hand_trial()
    report['hand_written_trial_s'] = timed(hand_trial, max(2, args.reps // 5))
    ag.train(env, 1, args.steps, L)
    report['fused_trial_s'] = timed(lambda: ag.train(env, 1, args.steps, L), max(2, args.reps // 5))
    report['trial_steps'] = args.steps
    print(json.dumps({k: report[k] for k in ('trial_steps', 'hand_written_trial_s', 'fused_trial_s')}), flush=True)
    print(json.dumps(report), flush=True)


if __name__ == '__main__':
    main()
