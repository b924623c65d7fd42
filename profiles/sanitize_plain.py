#!/usr/bin/env python
"""Small runs of the PLAIN (production) kernel instantiations for compute-sanitizer: the parity tests record traces and
therefore run the generic instantiations; this script runs the ones the benchmarks use, at sizes a sanitizer finishes
in seconds.  Usage: compute-sanitizer --tool memcheck|racecheck python profiles/sanitize_plain.py"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import cobel_rl_b200 as cb  # noqa: E402
from cobel_rl_b200 import agent as AG, memory as MEM  # noqa: E402
from cobel_rl_b200.interface import Gridworld, Topology  # noqa: E402
from cobel_rl_b200.misc.gridworld_tools import make_gridworld, make_open_field  # noqa: E402
from cobel_rl_b200.misc.topology_tools import linear_track  # noqa: E402
from cobel_rl_b200.policy import EpsilonGreedy  # noqa: E402


def main():
    dev = 'cuda:0'
    # Dyna-Q: 37 and 6 agents are fewer than two waves, so both runs use the warp-per-agent kernel (the
    # two-agents-per-warp kernel is selected from 2 * 7 * 4 agents per SM on)
    for n in (37, 6):
        st = cb.BatchStream(n, seed=1, device=dev)
        env = Gridworld(make_open_field(5, 5, 0, 1), rng=st)
        ag = AG.DynaQ(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=st))
        ag.train(env, 12, 30, 32)
    st = cb.BatchStream(9, seed=2, device=dev)
    env = Topology(*linear_track(10, 2, 1.0, 20.0, 'right'), rng=st)
    AG.QAgent(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=st), None, 0.9, 0.8, rng=st).train(env, 10, 30, 32)
    world = make_gridworld(6, 6, terminals=[5], rewards=[[5, 1.0]], starting_states=[30], invalid_transitions=[(1, 2), (2, 1)])
    st = cb.BatchStream(11, seed=3, device=dev)
    env = Gridworld(world, rng=st)
    mem = MEM.PMAMemory(world['sas'], EpsilonGreedy(0.1, rng=st), 0.9, 0.9, 0.9, 0.99, rng=st)
    pma = AG.PMA(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=st), mem, None, 0.9, 0.99)
    pma.mask_actions = True
    pma.train(env, 3, 40, 32)
    from cobel_rl_b200.memory.utils.metrics import DR
    w = make_open_field(8, 8, 0, 1)
    st = cb.BatchStream(5, seed=4, device=dev)
    env = Gridworld(w, rng=st)
    sm = MEM.SFMAMemory(DR(8, 8, w['sas'], 0.9, w['invalid_transitions']), env.n_states, 4, rng=st)
    sf = AG.SFMA(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=st), sm, None, 0.99, 0.99, rng=st)
    sf.mask_actions = True
    sf.train(env, 3, 60, 32)
    st = cb.BatchStream(4, seed=5, device=dev)
    env = Gridworld(make_open_field(6, 6, 0, 1), rng=st)
    AG.SR(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=st), None, 0.1, 0.99).train(env, 3, 30)
    torch.cuda.synchronize()
    print('sanitize_plain: done')


if __name__ == '__main__':
    main()
