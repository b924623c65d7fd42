#!/usr/bin/env python
"""SFMA train() on a 50x50 open field (2500 states, Euclidean similarity) with the memory options that need the fused
kernel, whose per-agent tables (485 KB with recency) then live in a device workspace (sfma_kernel<A, MODS, true>),
against the default options on the split path (sfma_step_kernel + sfma_replay_kernel).

Configurations: default (split path), recency, decay_strength = 0.95, reward_mod.  Each is timed with CUDA events
around one train() call of --agents agents (--trials x --steps, batch 32, eps 0.1) after a warm-up call of the same
configuration on 8 agents.  Prints the card and its power limit first, then one JSON line per configuration.
Usage: python profiles/sfma_large_options.py [--agents 4096] [--trials 2] [--steps 100]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cobel_rl_b200 as cb  # noqa: E402
from cobel_rl_b200.agent import SFMA  # noqa: E402
from cobel_rl_b200.interface import Gridworld  # noqa: E402
from cobel_rl_b200.memory import SFMAMemory  # noqa: E402
from cobel_rl_b200.memory.utils.metrics import Euclidean  # noqa: E402
from cobel_rl_b200.misc.gridworld_tools import make_open_field  # noqa: E402
from cobel_rl_b200.policy import EpsilonGreedy  # noqa: E402

CONFIGS = {'default (split path)': {}, 'recency': {'recency': True}, 'decay_strength=0.95': {'decay_strength': 0.95},
           'reward_mod': {'reward_mod': True}}


def timed_train(world, metric, n, seed, trials, steps, options):
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    env = Gridworld(world, rng=stream)
    mem = SFMAMemory(metric, 2500, 4, rng=stream)
    for k, v in options.items():
        setattr(mem, k, v)
    ag = SFMA(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream), mem, rng=stream)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    res = ag.train(env, trials, steps, 32)
    t1.record()
    torch.cuda.synchronize()
    sec = t0.elapsed_time(t1) / 1e3
    agent_steps = int(res['n_steps'].sum())
    out = {'seconds': sec, 'agent_steps': agent_steps, 'agent_steps_per_s': agent_steps / sec,
           'replayed': int(res['n_replay'].sum()), 'flags': int(res['flags'].abs().sum()),
           'workspace_bytes_per_agent': 0 if mem._workspace is None else mem._workspace.numel() // n}
    del ag, mem, env, stream, res
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--agents', type=int, default=4096)
    ap.add_argument('--trials', type=int, default=2)
    ap.add_argument('--steps', type=int, default=100)
    args = ap.parse_args()
    print(subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv'], capture_output=True,
                         text=True).stdout.strip(), flush=True)
    world = make_open_field(50, 50, 0, 1, dense_sas=False)
    metric = Euclidean(50, 50)
    for name, options in CONFIGS.items():
        timed_train(world, metric, 8, 1, 1, args.steps, options)                              # warm-up
        r = timed_train(world, metric, args.agents, 7, args.trials, args.steps, options)
        print(json.dumps({'config': name, 'world': '50x50', 'agents': args.agents, 'trials': args.trials,
                          'steps': args.steps, 'batch': 32, **r}), flush=True)


if __name__ == '__main__':
    main()
