#!/usr/bin/env python
"""bench.py -- headline benchmarks of the B200-native tabular simulator.

Metric (BASELINE.json): "agent-steps/sec incl. replay at 1/2/4/8 B200; PMA replay updates/sec".
The JSON line's top-level fields are the first metric on BASELINE.json configs[1]:
  4096 independent Dyna-Q agents per GPU (weak scaling) on the 5x5 open gridworld, the reference
  demo's setting (demo/gridworld/demo_dyna_q.py:36-56: 500 trials x <=50 steps, replay batch 32,
  epsilon 0.1, lr 0.99, gamma 0.99).  One "step" of the benchmark = one complete
  ``DynaQ.train(env, 500, 50, 32)`` of all agents from freshly initialised tables.
The second metric (PMA replay-updates/s on configs[2]: 10x10 walled gridworld, 16384 agents per
GPU) is measured in the same run and reported under the key "pma".  Other workloads
(--workload sfma|sr|q) print their own line with the same schema.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload dynaq|pma|sfma|sr|q]
                  [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  DESIGN.md "Measurement" documents every field.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# the CPU baseline runs one process per core: keep LAPACK single-threaded (must be set before NumPy loads)
os.environ.setdefault('OPENBLAS_NUM_THREADS', '1')
os.environ.setdefault('OMP_NUM_THREADS', '1')
os.environ.setdefault('MKL_NUM_THREADS', '1')

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SEED = 0x5EED
DUMP_BYTES = 60 * 1024 * 1024     # --dump-outputs: all arrays of one run together (under 64 MB with the .npy headers)

# Workloads.  bytes_per_unit = algorithmic bytes per unit (SURVEY.md section 8d, DESIGN.md).
WORKLOADS = {
    'dynaq': dict(
        desc='C2: 4096 Dyna-Q agents/GPU, 5x5 open field, 500 trials x <=50 steps, batch 32',
        metric='agent-steps/sec incl. replay', unit='agent-steps/s', kernel='dynaq_warp_kernel<4,PLAIN>',
        agents_per_gpu=4096, trials=500, steps=50, batch=32, world='open5', bytes_per_unit=2066,
        unit_key='n_steps', cpu_trials=500),
    'dynaq64k': dict(
        desc='Dyna-Q throughput regime: 65536 agents/GPU (two agents per warp), 5x5 open field, 500 trials x <=50 steps, batch 32',
        metric='agent-steps/sec incl. replay', unit='agent-steps/s', kernel='dynaq_pair_kernel<4>',
        agents_per_gpu=65536, trials=500, steps=50, batch=32, world='open5', bytes_per_unit=2066,
        unit_key='n_steps', cpu_trials=500, like='dynaq'),
    'pma': dict(
        desc='C3: 16384 PMA agents/GPU, 10x10 gridworld with walls, 4 trials x <=100 steps, replay batch 32 at '
             'trial start and end',
        metric='PMA replay updates/sec', unit='replay-updates/s', kernel='pma_main_kernel<4,PLAIN> + pma_band_factor_kernel + pma_sr_band_kernel<10> + pma_band_check_kernel',
        agents_per_gpu=16384, trials=4, steps=100, batch=32, world='walls10', bytes_per_unit=23 * 400 + 8 * 100,
        unit_key='n_replay', cpu_trials=4),
    'sfma': dict(
        desc='C4: 65536 SFMA agents/GPU, 20x20 open field, DR metric, default mode, 4 trials x <=200 steps, batch 32',
        metric='agent-steps/sec incl. replay', unit='agent-steps/s', kernel='sfma_step_kernel<4> + sfma_replay_kernel<4>',
        agents_per_gpu=65536, trials=4, steps=200, batch=32, world='open20', bytes_per_unit=138,
        unit_key='n_steps', cpu_trials=4),
    'sr': dict(
        desc='SR agents (dense S x S), 20x20 open field, 4096 agents/GPU, 4 trials x <=64 steps',
        metric='agent-steps/sec', unit='agent-steps/s', kernel='sr_tma_kernel<4>',
        agents_per_gpu=4096, trials=4, steps=64, batch=0, world='open20', bytes_per_unit=8 * 400 * 8 + 24,
        unit_key='n_steps', cpu_trials=4),
    'sr100': dict(
        desc='C5: SR agents with visited-set compaction, 100x100 open field, 1048576 agents in total (strong scaling: '
             'sharded over the GPUs), 2 trials x <=48 steps, max_visited 100',
        metric='agent-steps/sec', unit='agent-steps/s', kernel='sr_compact_kernel<4,PLAIN>',
        agents_total=1048576, trials=2, steps=48, batch=0, world='open100', bytes_per_unit=3 * 8 * 25 + 24,   # refined from the measured visited counts in measure()
        unit_key='n_steps', cpu_trials=2, scaling='strong', max_visited=100),
    'q': dict(
        desc='QAgent on the linear_track(10,2) topology graph, 4096 agents/GPU, 500 trials x <=50 steps, batch 32',
        metric='agent-steps/sec incl. replay', unit='agent-steps/s', kernel='q_warp_kernel<4,PLAIN>',
        agents_per_gpu=4096, trials=500, steps=50, batch=32, world='track', bytes_per_unit=2223,
        unit_key='n_steps', cpu_trials=500),
}


# agents per host core in the cpu_baseline leg: sized for roughly 10-20 s of CPU work per workload
CPU_AGENTS_PER_CORE = {'dynaq': 16, 'dynaq64k': 16, 'pma': 12, 'q': 16, 'sr': 8, 'sfma': 4, 'sr100': 1}


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs, burst copy)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def measured_traffic(name, agents_per_gpu):
    """DRAM bytes per launch of the workload's dominant kernel from the committed ncu capture
    (profiles/traffic.json), or None if no capture exists for this configuration."""
    try:
        t = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json'))).get(name)
    except (OSError, ValueError):
        return None
    if not t or t.get('agents_per_gpu') != agents_per_gpu:
        return None
    return t['bytes_per_launch']


def measured_issue(name, agents_per_gpu):
    """Warp-instructions per unit of the workload's kernels from the committed ncu counters (profiles/issue.json,
    written by profiles/collect_counters.py), or None if no capture exists for this configuration."""
    try:
        t = json.load(open(os.path.join(ROOT, 'profiles', 'issue.json'))).get(name)
    except (OSError, ValueError):
        return None
    if not t:
        return None
    if t.get('agents_per_gpu') != agents_per_gpu:      # instructions per unit barely depend on the number of agents
        t = dict(t, source='%s; counted at %d agents/GPU' % (t.get('source'), t.get('agents_per_gpu')))
    return t


# the bench worlds (the same definitions the parity cases use, oracle/cases.py; restated here so that the measured arm
# imports nothing from oracle/)
WALLS_10x10 = [(4, 5), (5, 4), (14, 15), (15, 14), (24, 25), (25, 24), (34, 35), (35, 34),
               (62, 72), (72, 62), (63, 73), (73, 63)]


def make_world(name):
    from cobel_rl_b200.misc.gridworld_tools import make_gridworld, make_open_field
    if name == 'open20':
        return make_open_field(20, 20, 0, 1)
    if name == 'open100':
        return make_open_field(100, 100, 0, 1, dense_sas=False)
    if name == 'open5':       # config C2, demo/gridworld/demo_dyna_q.py:41
        return make_gridworld(5, 5, terminals=[0], rewards=np.array([[0, 1]]), goals=[0])
    if name == 'walls10':     # config C3
        return make_gridworld(10, 10, terminals=[9], rewards=np.array([[9, 10]]), goals=[9], starting_states=[57],
                              invalid_transitions=WALLS_10x10)
    raise KeyError(name)


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            time.sleep(0.3)
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(smax) if smax else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


# --------------------------------------------------------------------------- #
# CPU baseline / reference arm: the reference's algorithm (oracle port) on host cores
# --------------------------------------------------------------------------- #

def reference_available():
    """The unmodified reference package (baseline/_ref, placed by oracle/install_reference.py) is importable."""
    try:
        from oracle import ref_loader
        return ref_loader.available()
    except Exception:
        return False


def _ref_worker(args):
    """One host core: a slice of agents run one after the other through the UNMODIFIED reference classes
    (cobel.agent.* from baseline/_ref, driven by the same per-agent uniform streams)."""
    name, agent_ids, trials = args
    os.environ['OPENBLAS_NUM_THREADS'] = '1'
    from oracle import ref_runs
    from oracle.philox import LazyStream
    wl = WORKLOADS[name]
    steps, batch = wl['steps'], wl['batch']
    units = 0
    if name == 'q':
        from cobel_rl_b200.misc.topology_tools import linear_track
        nodes, starts = linear_track(10, 2, 1.0, 20.0, 'right')
    else:
        world = make_world(wl['world'])
    for g in agent_ids:
        u = LazyStream(SEED, g)
        if name == 'dynaq':
            units += len(ref_runs.run_dynaq(world, u, trials, steps, batch)['states'])
        elif name == 'q':
            units += len(ref_runs.run_q_topology(nodes, starts, u, trials, steps, batch)['states'])
        elif name == 'sr':
            units += len(ref_runs.run_sr(world, u, trials, steps)['states'])
        elif name == 'sfma':
            from cobel_rl_b200.memory.utils.metrics import DR
            D = DR(world['width'], world['height'], world['sas'], 0.9, world['invalid_transitions']).D
            units += len(ref_runs.run_sfma(world, D, u, trials, steps, batch, mask_actions=True)['states'])
        elif name == 'pma':
            units += len(ref_runs.run_pma(world, u, trials, steps, batch, gamma_q=0.99, mask_actions=True)['replay'])
        else:
            raise ValueError(name)
    return units


def _cpu_worker(args):
    name, agent_ids, trials = args
    os.environ['OPENBLAS_NUM_THREADS'] = '1'
    from oracle import tabular as tb
    from oracle.philox import LazyStream
    wl = WORKLOADS[name]
    steps, batch = wl['steps'], wl['batch']
    if name == 'q':
        from cobel_rl_b200.misc.topology_tools import linear_track
        W = tb.compile_topology(*linear_track(10, 2, 1.0, 20.0, 'right'))
    else:
        world = make_world(wl['world'])
        if world['sas'] is None:
            W = {'S': world['states'], 'A': 4, 'succ': world['succ'], 'reward': world['rewards'].astype(np.float64),
                 'terminal': world['terminals'].astype(np.uint8), 'starts': world['starting_states'].astype(np.int32)}
        else:
            W = tb.compile_gridworld(world)
    S, A = W['S'], W['A']
    units = 0
    for g in agent_ids:
        rng = tb.Draws(LazyStream(SEED, g), 1)
        if name == 'dynaq':
            rec = tb.dynaq_train(W, tb.dynaq_init(S, A), rng, trials, steps, batch)
            units += len(rec.s)
        elif name == 'q':
            rec = tb.q_train(W, tb.q_init(S, A), rng, trials, steps, batch)
            units += len(rec.s)
        elif name in ('sr', 'sr100'):
            rec = tb.sr_train(W, tb.sr_init(S, A), rng, trials, steps)
            units += len(rec.s)
        elif name == 'sfma':
            from cobel_rl_b200.memory.utils.metrics import DR
            D = DR(world['width'], world['height'], world['sas'], 0.9, world['invalid_transitions']).D
            rec = tb.sfma_train(W, tb.sfma_init(S, A), D, rng, trials, steps, batch, mask_actions=True)
            units += len(rec.s)
        elif name == 'pma':
            st = tb.pma_init(tb.t0_from_succ(W['succ']), S, A)
            rec = tb.pma_train(W, st, rng, trials, steps, batch, gamma_q=0.99, mask_actions=True)
            units += len(rec.replay)
    return units


# agents per host core when the real reference runs (it is 2-3x slower than the vectorised oracle port)
REF_AGENTS_PER_CORE = {'dynaq': 6, 'pma': 4, 'q': 6, 'sr': 4, 'sfma': 2}


def cpu_run(name, agents_per_core=1, pool=None, cores=None, trials=None):
    """The reference's CPU loop, one process per host core, each running a slice of agents of the SAME workload
    (same world, hyper-parameters and per-agent streams): the UNMODIFIED reference (baseline/_ref) when it is
    present -- kind "reference" -- else the oracle port (kind "port"; always for sr100, whose dense tables do not
    exist in the reference's form)."""
    import multiprocessing as mp
    wl = WORKLOADS[name]
    trials = trials or wl['cpu_trials']
    cores = cores or os.cpu_count() or 1
    real = reference_available() and name in REF_AGENTS_PER_CORE
    worker = _ref_worker if real else _cpu_worker
    if real:
        agents_per_core = min(agents_per_core, REF_AGENTS_PER_CORE[name])
    ids = [list(range(c * agents_per_core, (c + 1) * agents_per_core)) for c in range(cores)]
    own = pool is None
    if own:
        pool = mp.get_context('spawn').Pool(cores)
        pool.map(worker, [('dynaq', [0], 1)] * cores)            # import / warm the workers
    t0 = time.perf_counter()
    units = sum(pool.map(worker, [(name, i, trials) for i in ids]))
    dt = time.perf_counter() - t0
    if own:
        pool.close()
    what = ('the unmodified reference classes (cobel.agent.* from baseline/_ref) under the same uniform streams'
            if real else 'oracle/tabular.py (NumPy restatement validated bit-exact against the reference)')
    return {'value': units / dt, 'unit': wl['unit'], 'cores': cores, 'kind': 'reference' if real else 'port',
            'sample': '%d agents (%d per core) of the same workload, %d trials x <=%d steps, batch %d: %d units in '
                      '%.1f s; %s' % (cores * agents_per_core, agents_per_core, trials, wl['steps'], wl['batch'],
                                      units, dt, what),
            'seconds': dt, 'units': units}


def run_reference(args):
    if int(os.environ.get('RANK', '0')) != 0:
        return
    import multiprocessing as mp
    name = args.workload
    wl = WORKLOADS[name]
    cores = os.cpu_count() or 1
    pool = mp.get_context('spawn').Pool(cores)
    pool.map(_ref_worker if (reference_available() and name in REF_AGENTS_PER_CORE) else _cpu_worker,
             [('dynaq', [0], 1)] * cores)
    for _ in range(args.warmup):
        cpu_run(name, 1, pool, cores)
    t_tot, u_tot, last = 0.0, 0, None
    for _ in range(args.steps):
        last = cpu_run(name, 1, pool, cores)
        t_tot += last['seconds']; u_tot += last['units']
    pool.close()
    val = u_tot / t_tot
    cb = {k: v for k, v in last.items() if k not in ('seconds', 'units')}
    cb['value'] = val
    print(json.dumps({
        'impl': 'reference', 'metric': wl['metric'], 'value': val, 'unit': wl['unit'],
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * t_tot / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': wl['desc'], 'note': 'each step = one agent per host core run through the workload '
                   '(%d trials)' % wl['cpu_trials']},
        'cpu_baseline': cb,
        'e2e': {'value': val, 'unit': wl['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }))


# --------------------------------------------------------------------------- #
# our arm
# --------------------------------------------------------------------------- #

class Job:
    """One workload on one rank: builds the agents through the public class API, exposes
    ``step()`` (kernel-only, inputs resident in HBM) and ``step_e2e()`` (host buffers in, results out)."""

    def __init__(self, name, dev, lo, n_local):
        import torch
        import cobel_rl_b200 as cb
        from cobel_rl_b200 import agent as AG, memory as MEM
        from cobel_rl_b200.interface import Gridworld, Topology
        from cobel_rl_b200.policy import EpsilonGreedy
        self.torch, self.wl, self.dev = torch, WORKLOADS[name], dev
        wl = self.wl
        self.name = name = wl.get('like', name)
        self.stream = st = cb.BatchStream(n_local, seed=SEED, device=dev, agent_id_base=lo)
        if name == 'q':
            from cobel_rl_b200.misc.topology_tools import linear_track
            self.env = Topology(*linear_track(10, 2, 1.0, 20.0, 'right'), rng=st)
        else:
            self.world = make_world(wl['world'])
            self.env = Gridworld(self.world, rng=st)
        env = self.env
        pol = EpsilonGreedy(0.1, rng=st)
        if name == 'dynaq':
            mem = MEM.DynaQMemory(env.n_states, 4, 0.9, rng=st)
            self.agent = AG.DynaQ(env.observation_space, env.action_space, pol, None, 0.99, 0.99, mem)
            self.state = {'Q': self.agent._Q, 'Mr': mem._rewards, 'Ms': mem._states, 'Mt': mem._terminals}
        elif name == 'q':
            self.agent = AG.QAgent(env.observation_space, env.action_space, pol, None, 0.9, 0.8, rng=st)
            self.agent._alloc_q(env.n_states)
            self.agent._ensure_log(wl['trials'] * wl['steps'])
            self.state = {'Q': self.agent._Q, 'log_len': self.agent._log_len}
        elif name == 'sr':
            self.agent = AG.SR(env.observation_space, env.action_space, pol, None, 0.1, 0.99)
            self.state = {'SR': self.agent._SR, 'rew': self.agent._rewards, 'model': self.agent._model}
        elif name == 'sr100':
            self.agent = AG.SR(env.observation_space, env.action_space, pol, None, 0.1, 0.99, compact=True,
                               max_visited=wl['max_visited'])
            # a fresh compact agent is just "nothing visited yet": rows are initialised on first visit
            self.state = {'n_visited': self.agent._n_visited}
        elif name == 'sfma':
            from cobel_rl_b200.memory.utils.metrics import DR
            w = self.world
            mem = MEM.SFMAMemory(DR(w['width'], w['height'], w['sas'], 0.9, w['invalid_transitions']),
                                 env.n_states, 4, rng=st)
            self.agent = AG.SFMA(env.observation_space, env.action_space, pol, mem, None, 0.99, 0.99, rng=st)
            self.agent.mask_actions = True
            self.state = {'Q': self.agent._Q, 'Mr': mem._rewards, 'Ms': mem._states, 'Mt': mem._terminals,
                          'C': mem._C, 'T': mem._T, 'I': mem._I}
        elif name == 'pma':
            mem = MEM.PMAMemory(self.world['sas'], EpsilonGreedy(0.1, rng=st), 0.9, 0.9, 0.9, 0.99, rng=st)
            self.agent = AG.PMA(env.observation_space, env.action_space, pol, mem, None, 0.9, 0.99)
            self.agent.mask_actions = True
            self.state = {'Q': self.agent._Q, 'Mr': mem._rewards, 'Ms': mem._states, 'Mt': mem._terminals,
                          'T': mem._T, 'SR': mem._SR}
        # per-agent state small enough to keep pristine device + pinned host copies of (everything except the
        # S x S matrices, which are re-broadcast on the device from one pristine matrix)
        # Tables whose initial content is the same for every agent (a fresh agent's zero Q table, the memory's initial
        # model, T and SR of the world) travel to the device as ONE template and are broadcast there; what differs per
        # agent (here: the stream positions; in a sweep also the hyper-parameter vectors) is uploaded per agent.
        same = {k: bool((v == v[0:1]).all().item()) for k, v in self.state.items()}
        self.big = {k: v[0].clone() for k, v in self.state.items() if same[k] and v.dim() >= 2}
        self.init = {k: v.clone() for k, v in self.state.items() if k not in self.big}
        self.host_in = {k: v.cpu().pin_memory() for k, v in self.init.items()}
        self.host_big = {k: v.cpu().pin_memory() for k, v in self.big.items()}
        self.host_draws = torch.ones(n_local, dtype=torch.int64).pin_memory()     # draw 0: the environment constructor
        tr = wl['trials']
        self.host_out = {'trial_steps': torch.empty((n_local, tr), dtype=torch.int32).pin_memory(),
                         'trial_reward': torch.empty((n_local, tr), dtype=torch.float64).pin_memory()}
        # the agent's tables after train(): what a caller reads back (a compact SR agent's are not all reset per step)
        a = self.agent
        self.tables = (dict(SRc=a._SRc, visited=a._visited, n_visited=a._n_visited, rew=a._rewards, model=a._model)
                       if name == 'sr100' else self.state)
        key = 'Q' if 'Q' in self.state else ('rew' if 'rew' in self.state else 'n_visited')
        self.out_key = key
        self.host_out[key] = torch.empty(self.state[key].shape, dtype=self.state[key].dtype).pin_memory()

    def _train(self):
        wl, a = self.wl, self.agent
        if self.name in ('sr', 'sr100'):
            return a.train(self.env, wl['trials'], wl['steps'])
        return a.train(self.env, wl['trials'], wl['steps'], wl['batch'])

    def reset(self):
        for k, v in self.init.items():
            self.state[k].copy_(v)
        for k, v in self.big.items():
            self.state[k].copy_(v.unsqueeze(0).expand_as(self.state[k]))
        self.stream.draw_count.fill_(1)        # draw 0 was consumed by the environment constructor

    def step(self):
        return self._train()

    def step_e2e(self):
        """Host buffers in (pinned), results out: per-agent tables + hyper-parameters H2D, train(), D2H."""
        for k, v in self.host_in.items():
            self.state[k].copy_(v, non_blocking=True)
        for k, v in self.host_big.items():
            self.state[k].copy_(v.to(self.dev, non_blocking=True).unsqueeze(0).expand_as(self.state[k]))
        self.stream.draw_count.copy_(self.host_draws, non_blocking=True)
        res = self._train()
        self.host_out[self.out_key].copy_(self.state[self.out_key], non_blocking=True)
        self.host_out['trial_steps'].copy_(res['trial_steps'], non_blocking=True)
        self.host_out['trial_reward'].copy_(res['trial_reward'], non_blocking=True)
        return res

    def outputs(self, res, budget):
        """The result of one train() and the agent's tables, on the host as float32 / float64 (integers exactly), for
        a fixed, seeded sample of this rank's agents sized to stay within ``budget`` bytes."""
        torch = self.torch
        n = self.stream.n_agents
        arrs = {k: v for k, v in res.items() if torch.is_tensor(v)}
        assert not set(arrs) & set(self.tables)
        arrs.update(self.tables)
        size = lambda v: 4 if v.dtype == torch.float32 else 8
        per_agent = 8 + sum(v[0].numel() * size(v) for v in arrs.values())     # + the agent id
        m = int(min(n, max(1, budget // per_agent)))
        ids = np.sort(np.random.default_rng(SEED).choice(n, m, replace=False))
        idx = torch.as_tensor(ids, device=self.dev)
        out = {'agents': (ids + self.stream.agent_id_base).astype(np.float64)}
        for k, v in arrs.items():
            a = v.index_select(0, idx).cpu().numpy()
            out[k] = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        return out

    def h2d_bytes(self):
        return sum(v.numel() * v.element_size() for v in list(self.host_in.values()) + list(self.host_big.values()) + [self.host_draws])

    def d2h_bytes(self):
        return sum(v.numel() * v.element_size() for v in self.host_out.values())


def measure(job, k, warmup, cdist, dev, flush, e2e=True, n_total=None, dump_budget=0):
    """Returns dict(ms kernel-only, ms e2e, per-rank units of one step, launches, wall), and with ``dump_budget`` the
    outputs of the last timed kernel-only step (``Job.outputs``)."""
    import torch
    from cobel_rl_b200 import _lib
    L = _lib.lib()

    def timed(fn, pre):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        res = None
        cdist.barrier(); torch.cuda.synchronize(dev)
        w0 = time.perf_counter()
        for s, e in evs:
            flush.fill_(1)                      # evict L2 (256 MiB write), outside the event pair
            if pre:
                pre()
            s.record()
            res = fn()
            e.record()
        torch.cuda.synchronize(dev); cdist.barrier()
        wall = time.perf_counter() - w0
        return [s.elapsed_time(e) for s, e in evs], wall, res

    for _ in range(max(warmup, 3)):
        job.reset(); job.step()
    torch.cuda.synchronize(dev)
    l0 = L.cobel_launch_count()
    ms, wall, res = timed(job.step, job.reset)
    launches = L.cobel_launch_count() - l0
    units = float(res[job.wl['unit_key']].sum().item())
    if job.name == 'sr100':
        # algorithmic bytes of a compact-SR step: rows SRc[s], SRc[s'] read and SRc[s] written over the V states
        # visited so far; V grows from 1 to the final count, so its mean over the run is taken as half of that
        vbar = 0.5 * float(job.agent._n_visited.double().mean().item())
        job.wl = dict(job.wl, bytes_per_unit=int(3 * 8 * vbar) + 24)
        WORKLOADS['sr100'] = job.wl
    if job.name == 'sfma':
        # per agent-step: 138 B of step work + the reactivations of the trial-end replay (8N + 24S + 61 B each,
        # DESIGN.md K5) spread over the steps actually taken
        S_, A_ = job.env.n_states, job.env.n_actions
        per_react = 8 * S_ * A_ + 24 * S_ + 61
        job.wl = dict(job.wl, bytes_per_unit=int(138 + per_react * float(res['n_replay'].sum().item()) /
                                                 max(float(res['n_steps'].sum().item()), 1.0)))
        WORKLOADS['sfma'] = job.wl
    out = {'ms': sum(ms) / len(ms), 'wall': wall, 'units': units, 'launches': int(launches), 'res': res,
           'steps_units': float(res['n_steps'].sum().item()), 'replay_units': float(res['n_replay'].sum().item())}
    if dump_budget:
        out['outputs'] = job.outputs(res, dump_budget)        # before the end-to-end steps overwrite the tables
    if e2e:
        for _ in range(2):
            job.step_e2e()
        torch.cuda.synchronize(dev)
        ms2, _, res2 = timed(job.step_e2e, None)
        assert float(res2[job.wl['unit_key']].sum().item()) == units
        out['ms_e2e'] = sum(ms2) / len(ms2)
        if n_total is not None:
            # the path's only collective: the final all-gather of the per-agent statistics (one NCCL call), warmed,
            # then timed inside the end-to-end step
            def e2e_gather():
                r = job.step_e2e()
                out['gathered'] = cdist.gather_results(r, n_total)
                return r
            for _ in range(2):
                e2e_gather()
            torch.cuda.synchronize(dev)
            ms3, _, _ = timed(e2e_gather, None)
            out['ms_e2e_gather'] = sum(ms3) / len(ms3)
    return out


def result_block(name, m, world, peak, peak_src, job, t_step, t_e2e, units_total, clocks=None):
    wl = WORKLOADS[name]
    achieved = wl['bytes_per_unit'] * m['units'] / (m['ms'] * 1e-3) / 1e9
    blk = {
        'metric': wl['metric'], 'value': units_total / (t_step * 1e-3), 'unit': wl['unit'], 'ms_per_step': t_step,
        'config': {'workload': wl['desc'], 'agents_total': wl['agents_per_gpu'] * world,
                   'units_per_bench_step': units_total,
                   'l2': 'flushed between steps with a 256 MiB write (outside the event pairs)',
                   'timing': 'CUDA events on the launching stream per step (table reset outside), mean of K, max over ranks',
                   'seed': SEED},
        'roofline': {'bound': 'hbm', 'kernel': wl['kernel'], 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                     'frac': achieved / peak, 'traffic': measured_traffic(name, wl['agents_per_gpu']),
                     'peak_source': peak_src,
                     'algorithmic_bytes_per_unit': wl['bytes_per_unit'],
                     'note': 'per-agent tables stay in shared memory for the whole launch, so DRAM traffic is far '
                             'below the algorithmic bytes; the kernels are issue / dependency-latency bound '
                             '(DESIGN.md, profiles/)'},
        'gpu_launches': m['launches'],
    }
    iss = measured_issue(name, wl['agents_per_gpu'])
    if iss:
        # what actually bounds these kernels: warp-instruction issue.  instr/unit from the committed ncu counters of
        # this configuration x the units of this run / (SM sub-partitions x SM clock x measured time)
        smsp = 4 * job.torch.cuda.get_device_properties(job.dev).multi_processor_count
        mhz = (clocks or {}).get('sm_mhz') or iss.get('sm_mhz') or 1965.0
        ipc = iss['warp_instr_per_unit'] * m['units'] / (smsp * mhz * 1e6 * m['ms'] * 1e-3)
        blk['roofline']['issue'] = {'warp_instr_per_unit': iss['warp_instr_per_unit'], 'achieved': ipc, 'peak': 1.0,
                                    'unit': 'warp-instructions/cycle/SM sub-partition', 'frac': ipc,
                                    'sm_mhz': mhz, 'source': iss.get('source')}
    if t_e2e is not None:
        blk['e2e'] = {'value': units_total / (t_e2e * 1e-3), 'unit': wl['unit'], 'h2d_bytes_per_step': job.h2d_bytes(),
                      'd2h_bytes_per_step': job.d2h_bytes(), 'ms_per_step': t_e2e,
                      'note': 'per step, from pinned host memory: one template of every table whose initial content is the '
                              'same for all agents (broadcast on the device) + the per-agent stream positions; back to '
                              'the host: the per-agent result table and per-trial statistics of ALL agents'}
    return blk


EXTRAS = ['pma', 'dynaq64k', 'q', 'sr', 'sfma', 'sr100']     # reported under their own keys next to the headline


def run_ours(args):
    import torch
    from cobel_rl_b200 import dist as cdist

    rank, world, local = cdist.init_from_env()
    assert world == args.gpus, 'launch with torchrun --nproc-per-node %d for --gpus %d' % (args.gpus, args.gpus)
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB L2
    peak, peak_src = peaks()
    names = [args.workload]
    if args.workload == 'dynaq' and not args.no_pma:
        names += ['pma'] if args.extras == 'pma' else (EXTRAS if args.extras == 'all' else [])
    blocks, head_clocks, dumps = {}, None, {}
    for name in names:
        wl = WORKLOADS[name]
        if wl.get('scaling') == 'strong':
            lo, hi = cdist.shard_range(wl['agents_total'], rank, world)
            n_local = hi - lo
            wl['agents_per_gpu'] = wl['agents_total'] // world
        else:
            n_local = wl['agents_per_gpu']
            lo, hi = cdist.shard_range(n_local * world, rank, world)
        n_total = int(cdist.sum_over_ranks(n_local, dev))
        job = Job(name, dev, lo, n_local)
        if args.profile_one:
            # one step between cudaProfilerStart / Stop (ncu --profile-from-start off): profiles/collect_counters.py
            for _ in range(max(args.warmup, 3)):
                job.reset(); job.step()
            job.reset()
            torch.cuda.synchronize(dev)
            torch.cuda.profiler.start()
            res = job.step()
            torch.cuda.synchronize(dev)
            torch.cuda.profiler.stop()
            print(json.dumps({'workload': name, 'agents_per_gpu': wl['agents_per_gpu'],
                              'units': float(res[wl['unit_key']].sum().item())}))
            return
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        m = measure(job, args.steps, args.warmup, cdist, dev, flush, n_total=n_total if world > 1 else None,
                    dump_budget=DUMP_BYTES // len(names) if args.dump_outputs and rank == 0 else 0)
        if 'outputs' in m:
            dumps[name] = m['outputs']
        clocks = sampler.stop() if rank == 0 else None
        if name == names[0]:
            head_clocks = clocks
        t_step = cdist.max_over_ranks(m['ms'], dev)
        t_e2e = cdist.max_over_ranks(m['ms_e2e'], dev)
        t_e2e_g = cdist.max_over_ranks(m['ms_e2e_gather'], dev) if 'ms_e2e_gather' in m else None
        if 'gathered' in m:
            assert m['gathered']['n_steps'].shape[0] == n_total
        units_total = cdist.sum_over_ranks(m['units'], dev)
        steps_total = cdist.sum_over_ranks(m['steps_units'], dev)
        replay_total = cdist.sum_over_ranks(m['replay_units'], dev)
        if rank == 0:
            blk = result_block(name, m, world, peak, peak_src, job, t_step, t_e2e, units_total, clocks)
            blk['config'].update(agent_steps_per_bench_step=steps_total, replay_updates_per_bench_step=replay_total,
                                 wall_s_incl_flush_and_reset=m['wall'])
            if t_e2e_g is not None:
                # e2e plus the final NCCL all-gather of the per-agent statistics (one collective, warmed)
                blk['e2e_with_gather'] = {'value': units_total / (t_e2e_g * 1e-3), 'unit': wl['unit'],
                                          'ms_per_step': t_e2e_g, 'gather_ms': t_e2e_g - t_e2e}
            blk['clocks'] = clocks
            blocks[name] = blk
        del job, m
        torch.cuda.empty_cache()
    if rank != 0:
        return
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arrs in dumps.items():
            for k, a in arrs.items():
                np.save(os.path.join(args.dump_outputs, '%s_%s.npy' % (name, k)), a)
    head = blocks[names[0]]
    out = {
        'metric': head['metric'], 'value': head['value'], 'unit': head['unit'], 'n_gpus': world,
        'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': head['ms_per_step'],
        'higher_is_better': True, 'scaling': WORKLOADS[names[0]].get('scaling', 'weak'), 'vs_baseline': None,
        'dtype': 'f64', 'data': 'synthetic', 'config': head['config'], 'roofline': head['roofline'], 'e2e': head['e2e'],
        'gpu_launches': head['gpu_launches'], 'clocks': head_clocks,
    }
    if 'e2e_with_gather' in head:
        out['e2e_with_gather'] = head['e2e_with_gather']
    if world == 1 and not args.no_cpu:
        cb = cpu_run(names[0], CPU_AGENTS_PER_CORE.get(names[0], 1))
        out['cpu_baseline'] = {k: v for k, v in cb.items() if k not in ('seconds', 'units')}
    for name in names[1:]:
        blk = blocks[name]
        if world == 1 and not args.no_cpu and name == 'pma':
            cb = cpu_run(name, CPU_AGENTS_PER_CORE.get(name, 1))
            blk['cpu_baseline'] = {k: v for k, v in cb.items() if k not in ('seconds', 'units')}
        blk['scaling'] = WORKLOADS[name].get('scaling', 'weak')
        out[name] = blk
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10, help='timed steps of every workload')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='dynaq', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--agents', type=int, default=0, help='override agents per GPU (profiling only; not the headline config)')
    ap.add_argument('--no-pma', action='store_true', help='headline workload only (no extra workloads)')
    ap.add_argument('--extras', default='all', choices=['all', 'pma', 'none'],
                    help='extra workloads reported under their own keys next to the Dyna-Q headline: all = PMA (the second '
                         'headline metric), Dyna-Q at 65536 agents, QAgent, dense SR, SFMA C4, compact SR C5')
    ap.add_argument('--profile-one', action='store_true', help='one step between cudaProfilerStart/Stop, for ncu')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step of each workload computed as DIR/<workload>_<name>.npy '
                         '(float32 / float64; a fixed, seeded sample of the agents of rank 0, at most 64 MB in all)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.agents:
        for w in WORKLOADS.values():
            w['agents_per_gpu'] = args.agents
            if 'agents_total' in w:
                w['agents_total'] = args.agents * args.gpus
            w['desc'] += ' [agents per GPU overridden to %d]' % args.agents
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == '__main__':
    main()
